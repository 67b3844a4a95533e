"""GPU parity of the front end (K4) against the CPU oracle: projection bytes, ring-ordered cloud, curvature and
labels bit-exact; feature index lists identical; VoxelGrid centroids bit-exact in xyz."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def pcl_points(cloud4):
    """Re-pack xyzi rows as 32-byte pcl::PointXYZI records (x y z pad intensity pad pad pad)."""
    out = np.zeros((len(cloud4), 8), np.float32)
    out[:, :3] = cloud4[:, :3]
    out[:, 4] = cloud4[:, 3]
    return out


@pytest.mark.parametrize("layout", ["packed16", "pcl32"])
def test_projection_bit_exact(ctx, oracle_mod, cfg_full, layout):
    cloud = cfg_full["cloud"].copy()
    # exercise the clamps: intensity above 255, a range just under / over 0.1 m, far ranges saturating at 255
    cloud[10] = [0.05, 0.02, 0.01, 300.0]
    cloud[11] = [0.099, 0.0, 0.01, 12.5]
    cloud[12] = [0.1, 0.0, 0.0, 255.5]
    cloud[13] = [40.0, 3.0, 1.0, 254.999]
    if layout == "pcl32":
        cloud = pcl_points(cloud)
    rng, inten, track = ctx.cloud_handler(cloud, 64, 1024)
    wr, wi, wt = oracle_mod.project(cloud, 64, 1024)
    assert np.array_equal(rng, wr)
    assert np.array_equal(inten, wi)
    assert np.array_equal(track, wt)
    assert rng.max() == 255 and (track[:, :3] == 0).all(1).any()


def _check_features(got, want):
    assert len(got["cloud"]) == len(want["cloud"]) > 1000
    assert np.array_equal(got["ring_start"], want["ring_start"]) and np.array_equal(got["ring_end"], want["ring_end"])
    assert np.array_equal(got["src_index"], want["src_index"])
    assert np.array_equal(got["cloud"][:, :3], want["cloud"][:, :3])
    # ring id is exact; relTime goes through atan2f whose last ulp differs between libm and CUDA
    assert np.array_equal(got["cloud"][:, 3].astype(np.int32), want["cloud"][:, 3].astype(np.int32))
    assert np.allclose(got["cloud"][:, 3], want["cloud"][:, 3], rtol=0, atol=1.6e-5)
    assert np.array_equal(got["curvature"], want["curvature"])
    assert np.array_equal(got["label"], want["label"])
    for k in ("sharp_idx", "less_sharp_idx", "flat_idx"):
        assert np.array_equal(got[k], want[k]), k
    assert got["less_flat"].shape == want["less_flat"].shape
    assert np.array_equal(got["less_flat"][:, :3], want["less_flat"][:, :3])
    assert np.allclose(got["less_flat"][:, 3], want["less_flat"][:, 3], rtol=0, atol=1.6e-5)


def test_feature_extraction_bit_exact_config1(ctx, oracle_mod, cfg_full):
    cloud = cfg_full["cloud"]
    got = ctx.extract_features(cloud, 0.3)
    want = oracle_mod.extract_features(cloud, 0.3)
    _check_features(got, want)
    assert (got["label"] == 2).sum() > 100 and (got["label"] == -1).sum() > 300


def test_feature_extraction_other_frames(ctx, oracle_mod, ilsm):
    """Different poses / seeds, a PCL-strided cloud and a frame with many dropped returns."""
    scene = ilsm.synth.Scene(1234, extent=60.0, n_boxes=25, n_poles=30)
    for k, (rv, t) in enumerate([([0, 0, 1.0], [3.0, -2.0, 1.2]), ([0.05, -0.03, -2.0], [-10.0, 8.0, 1.8])]):
        q = ilsm.synth.quat_from_rotvec(rv)
        cloud, _ = ilsm.synth.make_frame(scene, q, np.array(t), seed=77 + k, max_range=25.0 if k else 50.0)
        if k:
            cloud = pcl_points(cloud)
        _check_features(ctx.extract_features(cloud, 0.3), oracle_mod.extract_features(cloud, 0.3))


def test_feature_extraction_ragged(ctx, oracle_mod):
    """Tiny / empty inputs: rings shorter than the 6-point guard are skipped (scanRegistration.cpp:430)."""
    got = ctx.extract_features(np.zeros((0, 4), np.float32))
    assert len(got["cloud"]) == 0 and len(got["less_flat"]) == 0
    rng = np.random.default_rng(3)
    az = rng.uniform(-np.pi, np.pi, 40)
    pts = np.stack([5 * np.cos(az), 5 * np.sin(az), rng.uniform(-1.5, 1.5, 40), np.zeros(40)], 1).astype(np.float32)
    got = ctx.extract_features(pts)
    want = oracle_mod.extract_features(pts)
    assert np.array_equal(got["cloud"][:, :3], want["cloud"][:, :3]) and np.array_equal(got["label"], want["label"])
    assert len(got["sharp_idx"]) == len(want["sharp_idx"]) and len(got["less_flat"]) == len(want["less_flat"])


@pytest.mark.parametrize("leaf", [0.2, 0.4, 0.8])
def test_voxelgrid_bit_exact(ctx, oracle_mod, cfg_full, leaf):
    f = oracle_mod.extract_features(cfg_full["cloud"], 0.3)
    for cloud in (f["less_flat"], f["cloud"][f["less_sharp_idx"]], pcl_points(f["less_flat"][:3000])):
        got = ctx.voxelgrid(cloud, leaf)
        want = oracle_mod.voxelgrid(cloud, leaf)
        assert got.shape == want.shape and len(got) > 10
        assert np.array_equal(got, want)
    assert len(ctx.voxelgrid(np.zeros((0, 4), np.float32), leaf)) == 0
    one = np.array([[1.0, 2.0, 3.0, 7.0]], np.float32)
    assert np.array_equal(ctx.voxelgrid(one, leaf), one)


@pytest.mark.parametrize("n,leaf", [(2049, 0.2), (16384, 0.4), (16385, 0.4), (40000, 0.8), (65536, 0.2), (150000, 0.4)])
def test_voxelgrid_large_clouds_bit_exact(ctx, oracle_mod, ilsm, cfg_full, n, leaf):
    """More than 16384 points (mapOptimization filters ground + less-flat clouds of ~40k points, mapOptimization.cpp:
    368-370): the tiled multi-block sort path gives the same voxels, order and float centroids as the oracle.  2049 (the
    first hash-based size) and 16384 (the largest single block) are the block path's boundaries."""
    rng = np.random.default_rng(n)
    base = cfg_full["map_surf"]
    pts = np.zeros((n, 4), np.float32)
    pick = rng.integers(0, len(base), n)
    pts[:, :3] = base[pick, :3] + rng.normal(0, 0.05, (n, 3)).astype(np.float32)
    pts[:, 3] = rng.uniform(0, 64, n).astype(np.float32)
    pts[5, 0] = np.nan  # PCL skips non-finite points
    got = ctx.voxelgrid(pts, leaf)
    want = oracle_mod.voxelgrid(pts, leaf)
    assert got.shape == want.shape and len(got) > 1000
    assert np.array_equal(got, want)


def test_frame_to_pose_pipeline_matches_oracle(ctx, oracle_mod, ilsm, cfg_full):
    """Raw frame -> features -> stacks (0.4 / 0.8 VoxelGrid, laserMapping.cpp:608-616) -> registration, GPU vs oracle."""
    c = cfg_full
    f = ctx.extract_features(c["cloud"], 0.3)
    corner = ctx.voxelgrid(f["cloud"][f["less_sharp_idx"]], 0.4)
    surf = ctx.voxelgrid(f["less_flat"], 0.8)
    wf = oracle_mod.extract_features(c["cloud"], 0.3)
    wcorner = oracle_mod.voxelgrid(wf["cloud"][wf["less_sharp_idx"]], 0.4)
    wsurf = oracle_mod.voxelgrid(wf["less_flat"], 0.8)
    assert np.array_equal(corner[:, :3], wcorner[:, :3]) and np.array_equal(surf[:, :3], wsurf[:, :3])
    mc = ctx.new_map().set_input_cloud(c["map_corner"])
    ms = ctx.new_map().set_input_cloud(c["map_surf"])
    q, t, rep = ctx.register(mc, ms, corner, surf, c["q0"], c["t0"])
    wx, wsum, wnf = oracle_mod.register_aloam(c["map_corner"], c["map_surf"], wcorner, wsurf, np.concatenate([c["q0"], c["t0"]]))
    assert np.linalg.norm(t - wx[4:]) < 1e-4 and ilsm.synth.quat_angle(q, wx[:4]) < 1e-4
    assert rep.pass_[1].num_edge_factors == wnf[2] and rep.pass_[1].num_plane_factors == wnf[3]
    assert np.linalg.norm(t - c["t_true"]) < 0.05
    mc.close(), ms.close()


@pytest.mark.parametrize("name", ["open", "corridor", "fov22"])
def test_feature_extraction_matches_reference_code_golden(ctx, name):
    """The CUDA front end against outputs of the REFERENCE's own code (scanRegistration.cpp:227-589 compiled from the
    reference tree, tests/golden/make_golden_scanreg.py): ring-ordered cloud, ring bounds, curvature, labels and the four
    feature clouds, bit for bit on xyz (relTime differs from libm's atan2f by an ulp on the GPU and is compared to 1.6e-5
    elsewhere; it is unused downstream with DISTORTION 0)."""
    import os, sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    from make_golden_scanreg import CLOUDS, KEYS, as_reference_outputs, digest, frames
    gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "scanreg_reference.npz"))
    cloud = dict(frames())[name]
    assert digest(cloud) == str(gold[name + "/input_sha256"])
    got = as_reference_outputs(ctx.extract_features(cloud))
    for k in KEYS:
        assert tuple(gold[f"{name}/{k}/shape"]) == got[k].shape, (name, k)
        if k in CLOUDS:
            assert digest(np.ascontiguousarray(got[k][:, :3])) == str(gold[f"{name}/{k}/xyz_sha256"]), (name, k)
        else:
            assert digest(np.ascontiguousarray(got[k])) == str(gold[f"{name}/{k}/sha256"]), (name, k)





def test_projection_matches_reference_code_golden(ctx):
    """The CUDA projection against the outputs of the REFERENCE's own loop (image_handler.h_ouster:113-139 compiled from
    the reference tree, tests/golden/make_golden_imagehandler.py): range image, intensity image and cloud_track bit for bit."""
    import os, sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    from make_golden_imagehandler import digests, frame
    gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "imagehandler_reference.npz"))
    r = ctx.cloud_handler(frame())
    assert digests(r[0], r[1], r[2]) == [str(s) for s in gold["sha256"]]
