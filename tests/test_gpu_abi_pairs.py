"""Host and device forms of the C ABI pairs on a live context: both forms reject the same invalid arguments with the same
status and without a launch, the context keeps working afterwards, and one valid call of each form on the same input
gives the same bytes."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

OK, INVALID_ARG, NOT_ENOUGH_MAP, STATE = 0, -1, -4, -6


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def _dev(a):
    """A device copy of `a`, complete before the library's own stream reads it."""
    import torch
    d = torch.from_numpy(np.ascontiguousarray(a)).cuda()
    torch.cuda.synchronize()
    return d


def _zeros(shape, dtype):
    import torch
    d = torch.zeros(shape, dtype=dtype, device="cuda")
    torch.cuda.synchronize()
    return d


@pytest.fixture(scope="module")
def env():
    import torch
    import ilsm_b200 as ilsm
    ilsm._build.build()
    lib = ilsm.load_library()
    cfg = ilsm.synth.config1(n_map=20_000)
    ctx, other = ilsm.Context(0), ilsm.Context(0)
    e = dict(ilsm=ilsm, lib=lib, cfg=cfg, ctx=ctx, other=other)
    e["mc"] = ctx.new_map().set_input_cloud(cfg["map_corner"])
    e["ms"] = ctx.new_map().set_input_cloud(cfg["map_surf"])
    e["unbuilt_c"], e["unbuilt_s"] = ctx.new_map(), ctx.new_map()
    e["small_c"] = ctx.new_map().set_input_cloud(cfg["map_corner"][:10])  # at the corner guard (n must exceed 10)
    e["foreign"] = other.new_map().set_input_cloud(cfg["map_surf"])
    rng = np.random.default_rng(7)
    e["descs"] = rng.uniform(0, 2, (64, 1200)).astype(np.float32)
    e["sc"] = ilsm.ScanContextDb(ctx)
    e["sc"].add(e["descs"])
    torch.cuda.synchronize()
    yield e
    ctx.sync()
    for k in ("sc", "mc", "ms", "unbuilt_c", "unbuilt_s", "small_c", "foreign"):
        e[k].close()
    ctx.close(), other.close()


def same_status(e, host, dev):
    """Both forms return the same status and neither launches a kernel; returns that status."""
    lib = e["lib"]
    n0 = lib.ilsm_launch_count()
    rc_h = host()
    n1 = lib.ilsm_launch_count()
    rc_d = dev()
    e["ctx"].sync()
    n2 = lib.ilsm_launch_count()
    assert rc_h == rc_d, (rc_h, rc_d, lib.ilsm_last_error())
    assert n1 == n0 and n2 == n1, (n1 - n0, n2 - n1)
    return rc_h


def still_works(e):
    c = e["cfg"]
    idx, d2 = e["ms"].nearest_k_search(c["surf"][:64], 5)
    assert (idx >= 0).all() and np.isfinite(d2).all()


def test_map_build_and_knn_reject_alike(env):
    e, lib = env, env["lib"]
    pts = np.ascontiguousarray(e["cfg"]["surf"])
    d_pts = _dev(pts)
    m = e["ctx"].new_map()
    idx, d2 = np.zeros((64, 8), np.int32), np.zeros((64, 8), np.float32)
    d_idx, d_d2 = _dev(idx), _dev(d2)
    try:
        for n, stride in ((-1, 16), (4, 14), (4, 8)):
            assert same_status(e, lambda: lib.ilsm_map_build(m._h, _ptr(pts), n, stride, 0.0),
                               lambda: lib.ilsm_map_build_dev(m._h, d_pts.data_ptr(), n, stride, 0.0)) == INVALID_ARG
        assert lib.ilsm_map_build_pair_dev(m._h, d_pts.data_ptr(), -1, e["unbuilt_s"]._h, d_pts.data_ptr(), 4, 16, 0.0) == INVALID_ARG
        ms = e["ms"]
        for nq, stride, k in ((-1, 16, 5), (4, 14, 5), (4, 16, 0), (4, 16, 9)):
            assert same_status(e, lambda: lib.ilsm_knn(ms._h, _ptr(pts), nq, stride, k, 0.0, _ptr(idx), _ptr(d2)),
                               lambda: lib.ilsm_knn_dev(ms._h, d_pts.data_ptr(), nq, stride, k, 0.0, d_idx.data_ptr(),
                                                        d_d2.data_ptr())) == INVALID_ARG
        u = e["unbuilt_c"]
        assert same_status(e, lambda: lib.ilsm_knn(u._h, _ptr(pts), 4, 16, 5, 0.0, _ptr(idx), _ptr(d2)),
                           lambda: lib.ilsm_knn_dev(u._h, d_pts.data_ptr(), 4, 16, 5, 0.0, d_idx.data_ptr(),
                                                    d_d2.data_ptr())) == STATE
        still_works(e)
    finally:
        e["ctx"].sync()
        m.close()


def test_registration_pairs_reject_alike(env):
    e, lib, c = env, env["lib"], env["cfg"]
    corner, surf = np.ascontiguousarray(c["corner"]), np.ascontiguousarray(c["surf"])
    d_corner, d_surf = _dev(corner), _dev(surf)
    q, t = np.array(c["q0"]), np.array(c["t0"])
    qc, tc = q.copy(), t.copy()  # what a rejected host call would have overwritten
    d_pose = _dev(np.concatenate([q, t]))
    cloud = np.ascontiguousarray(c["cloud"])
    d_cloud = _dev(cloud)
    mc, ms, uc, us, small, foreign = (e[k] for k in ("mc", "ms", "unbuilt_c", "unbuilt_s", "small_c", "foreign"))
    cases = [  # (corner map, surf map, nc, stride, expected)
        (mc, ms, -1, 16, INVALID_ARG), (mc, ms, len(corner), 14, INVALID_ARG), (mc, foreign, len(corner), 16, INVALID_ARG),
        (uc, ms, len(corner), 16, STATE), (mc, us, len(corner), 16, STATE), (small, ms, len(corner), 16, NOT_ENOUGH_MAP),
    ]
    for a, b, nc, stride, want in cases:
        assert same_status(
            e, lambda: lib.ilsm_register(e["ctx"]._h, a._h, b._h, _ptr(corner), nc, _ptr(surf), len(surf), stride, _ptr(qc),
                                         _ptr(tc), None, None),
            lambda: lib.ilsm_register_dev(e["ctx"]._h, a._h, b._h, d_corner.data_ptr(), nc, d_surf.data_ptr(), len(surf), stride,
                                          d_pose.data_ptr(), None, None)) == want, (a, b, nc, stride)
        if want != NOT_ENOUGH_MAP:  # the association applies no map-size guard
            assert same_status(
                e, lambda: lib.ilsm_associate(e["ctx"]._h, a._h, b._h, _ptr(corner), nc, _ptr(surf), len(surf), stride, _ptr(q),
                                              _ptr(t), None, None, None, None),
                lambda: lib.ilsm_associate_dev(e["ctx"]._h, a._h, b._h, d_corner.data_ptr(), nc, d_surf.data_ptr(), len(surf),
                                               stride, d_pose.data_ptr(), None)) == want, (a, b, nc, stride)
    frame_cases = [  # (corner map, surf map, n, stride, line_res, expected)
        (mc, ms, -1, 16, 0.4, INVALID_ARG), (mc, ms, len(cloud), 12, 0.4, INVALID_ARG), (mc, ms, len(cloud), 16, 0.0, INVALID_ARG),
        (mc, foreign, len(cloud), 16, 0.4, INVALID_ARG), (uc, ms, len(cloud), 16, 0.4, STATE), (mc, us, len(cloud), 16, 0.4, STATE),
        (small, ms, len(cloud), 16, 0.4, NOT_ENOUGH_MAP),
    ]
    for a, b, n, stride, lr, want in frame_cases:
        assert same_status(
            e, lambda: lib.ilsm_register_frame(e["ctx"]._h, a._h, b._h, _ptr(cloud), n, stride, 0.3, lr, 0.8, _ptr(qc),
                                               _ptr(tc), None, None, None),
            lambda: lib.ilsm_register_frame_dev(e["ctx"]._h, a._h, b._h, d_cloud.data_ptr(), n, stride, 0.3, lr, 0.8,
                                                d_pose.data_ptr(), None)) == want, (a, b, n, stride, lr)
    assert np.array_equal(d_pose.cpu().numpy(), np.concatenate([q, t]))  # no rejected call touched the pose
    still_works(e)


def test_register_frame_unbuilt_maps_without_size_guard(env):
    """The map-size guard off (host form) or at its defaults (device form): an unbuilt map is still refused before any
    launch."""
    e, lib, c = env, env["lib"], env["cfg"]
    ilsm = e["ilsm"]
    cloud = np.ascontiguousarray(c["cloud"])
    d_cloud = _dev(cloud)
    q, t = np.array(c["q0"]), np.array(c["t0"])
    qc, tc = q.copy(), t.copy()  # what a rejected host call would have overwritten
    d_pose = _dev(np.concatenate([q, t]))
    off = ilsm.RegOpts()
    lib.ilsm_reg_opts_default(C.byref(off))
    off.min_corner_map = off.min_surf_map = 0
    for a, b in ((e["unbuilt_c"], e["ms"]), (e["mc"], e["unbuilt_s"]), (e["unbuilt_c"], e["unbuilt_s"])):
        assert same_status(
            e, lambda: lib.ilsm_register_frame(e["ctx"]._h, a._h, b._h, _ptr(cloud), len(cloud), 16, 0.3, 0.4, 0.8, _ptr(qc),
                                               _ptr(tc), C.byref(off), None, None),
            lambda: lib.ilsm_register_frame_dev(e["ctx"]._h, a._h, b._h, d_cloud.data_ptr(), len(cloud), 16, 0.3, 0.4, 0.8,
                                                d_pose.data_ptr(), None)) == STATE
        assert b"map not built" in lib.ilsm_last_error()
    still_works(e)


def test_frontend_and_lm_pairs_reject_alike(env):
    e, lib, ctx = env, env["lib"], env["ctx"]
    ilsm = e["ilsm"]
    cloud = np.ascontiguousarray(e["cfg"]["cloud"])
    d_cloud = _dev(cloud)
    rng_img, inten, track = np.zeros(len(cloud), np.uint8), np.zeros(len(cloud), np.uint8), np.zeros((len(cloud), 4), np.float32)
    d_rng, d_inten, d_track = _dev(rng_img), _dev(inten), _dev(track)
    for H, W, stride in ((0, 1024, 16), (64, -1, 16), (64, 1024, 12), (64, 1024, 14)):
        assert same_status(e, lambda: ctx._lib.ilsm_project(ctx._h, _ptr(cloud), H, W, stride, _ptr(rng_img), _ptr(inten), _ptr(track)),
                           lambda: lib.ilsm_project_dev(ctx._h, d_cloud.data_ptr(), H, W, stride, d_rng.data_ptr(), d_inten.data_ptr(),
                                                        d_track.data_ptr())) == INVALID_ARG
    good = ilsm.Pc2Layout()
    lib.ilsm_pc2_layout_pcl_xyzi(C.byref(good))
    short, odd_type = ilsm.Pc2Layout(), ilsm.Pc2Layout()
    lib.ilsm_pc2_layout_pcl_xyzi(C.byref(short))
    short.point_step = 10
    lib.ilsm_pc2_layout_pcl_xyzi(C.byref(odd_type))
    odd_type.intensity_datatype = 3
    blob = np.zeros(len(cloud) * 32, np.uint8)
    d_blob = _dev(blob)
    for n, lay in ((-1, good), (16, short), (16, odd_type)):
        assert same_status(e, lambda: lib.ilsm_pc2_pack(ctx._h, _ptr(cloud), n, C.byref(lay), _ptr(blob)),
                           lambda: lib.ilsm_pc2_pack_dev(ctx._h, d_cloud.data_ptr(), n, C.byref(lay), d_blob.data_ptr())) == INVALID_ARG
        assert same_status(e, lambda: lib.ilsm_pc2_unpack(ctx._h, _ptr(blob), n, C.byref(lay), _ptr(track)),
                           lambda: lib.ilsm_pc2_unpack_dev(ctx._h, d_blob.data_ptr(), n, C.byref(lay), d_track.data_ptr())) == INVALID_ARG
    cost, H6, g6 = C.c_double(), np.zeros(36), np.zeros(6)
    q, t = np.array(e["cfg"]["q0"]), np.array(e["cfg"]["t0"])
    d_pose = _dev(np.concatenate([q, t]))
    assert same_status(e, lambda: lib.ilsm_eval_normal_eq(ctx._h, _ptr(q), _ptr(t), 0.1, C.byref(cost), None, _ptr(g6)),
                       lambda: lib.ilsm_eval_normal_eq_dev(ctx._h, d_pose.data_ptr(), 0.1, None)) == INVALID_ARG
    still_works(e)


def test_scancontext_pairs_reject_alike(env):
    e, lib = env, env["lib"]
    sc = e["sc"]
    n_db = len(sc)
    descs = np.zeros((4097, 1200), np.float32)
    descs[:len(e["descs"])] = e["descs"]
    d_descs = _dev(descs)
    dist, ids, sh = np.zeros(4097 * 17), np.zeros(4097 * 17, np.int32), np.zeros(4097 * 17, np.int32)
    d_dist, d_ids, d_sh = _dev(dist), _dev(ids), _dev(sh)
    d_packed = _dev(np.zeros(4097 * 16 * 17, np.uint8))
    assert same_status(e, lambda: lib.ilsm_sc_add(sc._h, _ptr(descs), -1),
                       lambda: lib.ilsm_sc_add_dev(sc._h, d_descs.data_ptr(), -1)) == INVALID_ARG
    for n_search, k in ((-1, 0), (-1, 17), (n_db + 1, 5)):
        assert same_status(e, lambda: lib.ilsm_sc_query_topk(sc._h, _ptr(descs), n_search, 0, k, _ptr(dist), _ptr(ids), _ptr(sh)),
                           lambda: lib.ilsm_sc_query_topk_dev(sc._h, d_descs.data_ptr(), n_search, 0, k, d_dist.data_ptr(),
                                                              d_ids.data_ptr(), d_sh.data_ptr())) == INVALID_ARG
    for nq, k in ((0, 5), (4097, 5), (2, 0), (2, 17)):
        for host, dev in ((lib.ilsm_sc_query_topk_batch, lib.ilsm_sc_query_topk_batch_dev),
                          (lib.ilsm_sc_query_topk_sharded, lib.ilsm_sc_query_topk_sharded_dev)):
            assert same_status(e, lambda: host(sc._h, _ptr(descs), nq, -1, 0, k, _ptr(dist), _ptr(ids), _ptr(sh)),
                               lambda: dev(sc._h, d_descs.data_ptr(), nq, -1, 0, k, d_packed.data_ptr())) == INVALID_ARG, (nq, k)
    assert len(sc) == n_db
    _, i, _ = sc.query_topk(e["descs"][3], k=5)
    assert i[0] == 3


def _unpack(packed, B, k):
    rec = np.frombuffer(packed.tobytes(), np.uint8).reshape(B, 16 * k)
    return (rec[:, :8 * k].copy().view(np.float64), rec[:, 8 * k:12 * k].copy().view(np.int32),
            rec[:, 12 * k:16 * k].copy().view(np.int32))


def test_forms_give_the_same_bytes(env):
    """One valid call of each form on the same input, for the pairs no other test compares."""
    import torch
    e, lib, c, ctx = env, env["lib"], env["cfg"], env["ctx"]
    ilsm = e["ilsm"]
    # map build: the host-built and the device-built map hold the same points and answer k-NN alike
    pts = np.ascontiguousarray(c["map_surf"])
    d_pts = _dev(pts)
    a, b = ctx.new_map().set_input_cloud(pts), ctx.new_map().build_dev(d_pts.data_ptr(), len(pts), 12)
    ctx.sync()
    queries = np.ascontiguousarray(c["surf"])
    assert np.array_equal(a.points(), b.points())
    ia, da = a.nearest_k_search(queries, 5)
    ib, db = b.nearest_k_search(queries, 5)
    assert np.array_equal(ia, ib) and np.array_equal(da, db)
    ctx.sync()
    a.close(), b.close()
    # k-NN
    d_q, d_idx, d_d2 = _dev(queries), _zeros((len(queries), 5), torch.int32), _zeros((len(queries), 5), torch.float32)
    e["ms"].knn_dev(d_q.data_ptr(), len(queries), 16, 5, 0.0, d_idx.data_ptr(), d_d2.data_ptr())
    ctx.sync()
    ih, dh = e["ms"].nearest_k_search(queries, 5)
    assert np.array_equal(ih, d_idx.cpu().numpy()) and np.array_equal(dh, d_d2.cpu().numpy())
    # association: the same factors, seen through the evaluation at the same pose
    corner, surf = np.ascontiguousarray(c["corner"]), np.ascontiguousarray(c["surf"])
    pose0 = np.concatenate([c["q0"], c["t0"]])
    d_corner, d_surf, d_pose = _dev(corner), _dev(surf), _dev(pose0)
    ctx.associate(e["mc"], e["ms"], corner, surf, c["q0"], c["t0"])
    eh = ctx.eval_normal_eq(c["q0"], c["t0"])
    ctx.associate_dev(e["mc"], e["ms"], d_corner.data_ptr(), len(corner), d_surf.data_ptr(), len(surf), 16, d_pose.data_ptr())
    ed = ctx.eval_normal_eq(c["q0"], c["t0"])
    assert eh[0] == ed[0] and np.array_equal(eh[1], ed[1]) and np.array_equal(eh[2], ed[2])
    # frame registration: the pose after the host form equals the pose the device form leaves in place
    cloud = np.ascontiguousarray(c["cloud"])
    d_cloud = _dev(cloud)
    qh, th, _, _ = ctx.register_frame(e["mc"], e["ms"], cloud, c["q0"], c["t0"])
    ctx.register_frame_dev(e["mc"], e["ms"], d_cloud.data_ptr(), len(cloud), 16, d_pose.data_ptr())
    ctx.sync()
    assert np.concatenate([qh, th]).tobytes() == d_pose.cpu().numpy().tobytes()
    # projection
    rh, ih_, trh = ctx.cloud_handler(cloud)
    d_r, d_i, d_t = _zeros(len(cloud), torch.uint8), _zeros(len(cloud), torch.uint8), _zeros((len(cloud), 4), torch.float32)
    ctx.project_dev(d_cloud.data_ptr(), 64, 1024, 16, d_r.data_ptr(), d_i.data_ptr(), d_t.data_ptr())
    ctx.sync()
    assert np.array_equal(rh.ravel(), d_r.cpu().numpy()) and np.array_equal(ih_.ravel(), d_i.cpu().numpy())
    assert np.array_equal(trh, d_t.cpu().numpy())
    # PointCloud2 pack / unpack
    lay = ilsm.Pc2Layout()
    lib.ilsm_pc2_layout_pcl_xyzi(C.byref(lay))
    blob = ctx.pc2_pack(cloud, lay)
    d_blob_out = _zeros(len(blob), torch.uint8)
    assert lib.ilsm_pc2_pack_dev(ctx._h, d_cloud.data_ptr(), len(cloud), C.byref(lay), d_blob_out.data_ptr()) == OK
    ctx.sync()
    assert np.array_equal(blob, d_blob_out.cpu().numpy())
    back = ctx.pc2_unpack(blob, lay)
    d_blob, d_back = _dev(blob), _zeros((len(cloud), 4), torch.float32)
    assert lib.ilsm_pc2_unpack_dev(ctx._h, d_blob.data_ptr(), len(cloud), C.byref(lay), d_back.data_ptr()) == OK
    ctx.sync()
    assert back.tobytes() == d_back.cpu().numpy().tobytes()
    # ScanContext: a database filled by each add form, then the query forms
    descs = e["descs"]
    d_descs = _dev(descs)
    s1, s2 = ilsm.ScanContextDb(ctx), ilsm.ScanContextDb(ctx)
    s1.add(descs)
    s2.add_dev(d_descs.data_ptr(), len(descs))
    ctx.sync()
    q = np.ascontiguousarray(descs[5] + 0.01)
    r1, r2 = s1.query_topk(q, k=10), s2.query_topk(q, k=10)
    assert all(np.array_equal(x, y) for x, y in zip(r1, r2))
    d_qd = _dev(q)
    d_dist, d_id, d_sh = _zeros(10, torch.float64), _zeros(10, torch.int32), _zeros(10, torch.int32)
    s1.query_topk_dev(d_qd.data_ptr(), 10, -1, 0, d_dist.data_ptr(), d_id.data_ptr(), d_sh.data_ptr())
    ctx.sync()
    assert np.array_equal(r1[0], d_dist.cpu().numpy()) and np.array_equal(r1[1], d_id.cpu().numpy())
    assert np.array_equal(r1[2], d_sh.cpu().numpy())
    qs = np.ascontiguousarray(descs[:6] + 0.01)
    d_qs = _dev(qs)
    for host, dev in ((s1.query_topk_batch, lib.ilsm_sc_query_topk_batch_dev),
                      (s1.query_topk_sharded, lib.ilsm_sc_query_topk_sharded_dev)):
        hd, hi, hs = host(qs, k=7, id_offset=100)
        d_packed = _zeros(len(qs) * 16 * 7, torch.uint8)
        assert dev(s1._h, d_qs.data_ptr(), len(qs), -1, 100, 7, d_packed.data_ptr()) == OK
        ctx.sync()
        dd, di, ds = _unpack(d_packed.cpu().numpy(), len(qs), 7)
        assert np.array_equal(hd, dd) and np.array_equal(hi, di) and np.array_equal(hs, ds)
    ctx.sync()
    s1.close(), s2.close()
