"""GPU parity of the full per-frame loop (scanRegistration -> laserOdometry -> laserMapping, BASELINE config 2) against
the CPU oracle chained the same way, on a short synthetic corridor sequence."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def corridor_frames(S, n_frames, seed0=0x5EED0010):
    """SURVEY 8d config 2: 3 m x 3 m corridor with pillars every 5 m, 0.2 m/frame forward + sinusoidal yaw +-5 deg."""
    scene = S.Scene(corridor=True, length=120.0)
    out = []
    for k in range(n_frames):
        yaw = np.deg2rad(5.0) * np.sin(2 * np.pi * k / 50.0)
        q = S.quat_from_rotvec([0.0, 0.0, yaw])
        t = np.array([2.0 + 0.2 * k, 0.1 * np.sin(k / 15.0), 1.2])
        cloud, _ = S.make_frame(scene, q, t, seed=seed0 + k)
        out.append((cloud, q, t))
    return out


def rel_pose(S, q0, t0, q, t):
    """Pose of frame k in the frame of frame 0 (the SLAM world is the first sensor frame)."""
    R0 = S.quat_to_mat(q0)
    return S.quat_mul(S.quat_inv(q0), q), R0.T @ (t - t0)


def test_sequence_matches_oracle(ctx, oracle_mod, ilsm):
    S = ilsm.synth
    frames = corridor_frames(S, 12)
    slam = ilsm.Slam(ctx, 0.4, 0.8, 0.3, 8192)
    oslam = oracle_mod.Slam(0.4, 0.8, 0.3)
    q0, t0 = frames[0][1], frames[0][2]
    for k, (cloud, q, t) in enumerate(frames):
        gqo, gto, gqm, gtm, st = slam.frame(cloud)
        wodom, wmap, info = oslam.frame(cloud)
        f = info["features"]
        # front end: the five published clouds have identical sizes (labels are bit-exact, tested in test_gpu_frontend)
        assert (st.n_cloud, st.n_sharp, st.n_less_sharp, st.n_flat, st.n_less_flat) == \
               (len(f["cloud"]), len(f["sharp_idx"]), len(f["less_sharp_idx"]), len(f["flat_idx"]), len(f["less_flat"]))
        assert st.ran_odometry == (1 if k > 0 else 0)
        # odometry and mapped poses: 1e-4 m / 1e-4 rad (north-star bar)
        assert np.linalg.norm(gto - wodom[4:]) < 1e-4 and S.quat_angle(gqo, wodom[:4]) < 1e-4, k
        assert np.linalg.norm(gtm - wmap[4:]) < 1e-4 and S.quat_angle(gqm, wmap[:4]) < 1e-4, k
        wst = info["cubemap"]
        assert st.cubemap.ran_optimization == wst.ran_optimization
        assert (st.cubemap.n_map_corner, st.cubemap.n_map_surf, st.cubemap.n_stack_corner, st.cubemap.n_stack_surf) == \
               (wst.n_map_corner, wst.n_map_surf, wst.n_stack_corner, wst.n_stack_surf), k
        if k > 0:
            for p in range(2):
                assert st.odometry.pass_[p].num_edge_factors + st.odometry.pass_[p].num_plane_factors == \
                       int(info["odometry"][1][2 * p] + info["odometry"][1][2 * p + 1])
        # and the estimate tracks the ground truth (the corridor is well constrained except along its axis)
        qr, tr = rel_pose(S, q0, t0, q, t)
        if k > 1:
            assert np.linalg.norm(gtm - tr) < 0.3, (k, gtm, tr)
    # the map itself: every occupied cube of the oracle's window is identical on the device (this also joins the
    # insertion of the last frame, which the pipeline defers to its side stream)
    view = slam.cubemap()
    occupied = [i for i in range(4851) if len(oslam.cube.cube(1, i)) or len(oslam.cube.cube(0, i))]
    assert len(occupied) >= 2
    n_pts = 0
    for idx in occupied:
        for which in (0, 1):
            g, w = view.cube(which, idx), oslam.cube.cube(which, idx)
            # xyz bit-exact; the intensity channel carries scanID + 0.1 * relTime, whose atan2f is libm on the CPU and
            # CUDA's on the GPU (1 ulp apart now and then; unused downstream with DISTORTION 0, SURVEY 8a row a3)
            assert g.shape == w.shape and np.array_equal(g[:, :3], w[:, :3]), (idx, which)
            assert np.allclose(g[:, 3], w[:, 3], rtol=0, atol=1e-5), (idx, which)
            n_pts += len(g)
    assert n_pts > 1500
    slam.close()


def test_fork_mode_skips_odometry_optimisation(ctx, oracle_mod, ilsm):
    """use_aloam = 0 (frame not flagged "skip_intensity", laserOdometry.cpp:406-417): the stale q/t_last_curr is still
    composed; GPU and oracle agree."""
    S = ilsm.synth
    frames = corridor_frames(S, 5)
    slam = ilsm.Slam(ctx, 0.4, 0.8, 0.3, 8192)
    oslam = oracle_mod.Slam(0.4, 0.8, 0.3)
    flags = [True, True, False, False, True]
    for (cloud, _, _), fl in zip(frames, flags):
        gqo, gto, gqm, gtm, st = slam.frame(cloud, use_aloam=fl)
        wodom, wmap, info = oslam.frame(cloud, use_aloam=fl)
        assert np.linalg.norm(gto - wodom[4:]) < 1e-4 and S.quat_angle(gqo, wodom[:4]) < 1e-4
        assert np.linalg.norm(gtm - wmap[4:]) < 1e-4 and S.quat_angle(gqm, wmap[:4]) < 1e-4
    assert st.ran_odometry == 1
    slam.close()


def test_launched_pipeline_with_mapoptimization_matches_oracle(ctx, oracle_mod, ilsm):
    """spot.launch starts scanRegistration + laserOdometry + the mapOptimization node: the same loop with the ground-map
    mapping stage (ground extraction from the frame already on the device), over open ground."""
    S = ilsm.synth
    scene = S.Scene(S.SEED_MAP)
    q0, t0 = S.default_pose()
    slam = ilsm.Slam(ctx, min_range=0.3, mapping="mapOptimization")
    oslam = oracle_mod.Slam(min_range=0.3, mapping="mapOptimization")
    for k in range(6):
        q = S.quat_mul(q0, S.quat_from_rotvec([0, 0, 0.02 * k]))
        t = t0 + np.array([0.25 * k, 0.05 * k, 0.0])
        cloud, _ = S.make_frame(scene, q, t, seed=700 + k)
        gqo, gto, gqm, gtm, st = slam.frame(cloud)
        wodom, wmap, info = oslam.frame(cloud)
        assert np.linalg.norm(gto - wodom[4:]) < 1e-4 and S.quat_angle(gqo, wodom[:4]) < 1e-4, k
        assert np.linalg.norm(gtm - wmap[4:]) < 1e-4 and S.quat_angle(gqm, wmap[:4]) < 1e-4, k
        mi = info["mapopt"]
        assert st.cubemap.ran_optimization == mi["ran_optimization"] == (1 if k else 0)
        assert st.cubemap.n_map_surf == mi["map_size"]
        if k:
            assert st.cubemap.n_stack_surf == mi["n_query"] and bool(st.cubemap.n_valid) == mi["converged"]
            assert st.mapping.pass_[0].num_plane_factors == mi["n_plane_factors"]
    slam.close()


@pytest.mark.parametrize("mapping", ["laserMapping", "mapOptimization"])
def test_pipeline_survives_degenerate_frames(ctx, ilsm, mapping):
    """No-return frames (all zeros), NaN points and an empty cloud must not fault: the reference's guards (feature
    counts, map-size guard of laserMapping.cpp:624, RANSAC with < 3 band points) all have device-side equivalents."""
    S = ilsm.synth
    scene = S.Scene(corridor=True, length=60.0)
    slam = ilsm.Slam(ctx, 0.4, 0.8, 0.3, 4096, mapping=mapping)
    zeros = np.zeros((65536, 4), np.float32)
    qo, to, qm, tm, st = slam.frame(zeros)                      # nothing but no-returns
    assert st.n_cloud == 0 and np.all(np.isfinite(tm)) and np.all(np.isfinite(qm))
    q = S.quat_from_rotvec([0, 0, 0.0])
    good, _ = S.make_frame(scene, q, np.array([2.0, 0.0, 1.2]), seed=1)
    qo, to, qm, tm, st = slam.frame(good)
    assert st.n_cloud > 10000 and np.all(np.isfinite(tm))
    bad = good.copy()
    bad[::7, :3] = np.nan                                        # NaN returns sprinkled over the frame
    qo, to, qm, tm, st = slam.frame(bad)
    assert np.all(np.isfinite(tm)) and np.all(np.isfinite(qm)) and np.all(np.isfinite(to))
    qo, to, qm, tm, st = slam.frame(zeros)                      # and an empty frame in the middle of a run
    assert np.all(np.isfinite(tm))
    qo, to, qm, tm, st = slam.frame(good)
    assert np.all(np.isfinite(tm)) and st.n_cloud > 10000
    qo, to, qm, tm, st = slam.frame(np.zeros((0, 4), np.float32))
    assert st.n_cloud == 0
    slam.close()


def test_pipelined_mapping_stage_gives_the_same_poses(ctx, ilsm):
    """ilsm_slam_create_async: laserMapping as its own stage on a second context (frame k's mapping overlaps frame k+1's
    front end + odometry).  Odometry poses frame for frame and mapped poses one call later are bit-identical to the
    synchronous loop -- also when some frames skip the odometry solve (use_aloam = 0); misuse of the two handle kinds is
    rejected."""
    import os, sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    from sequence_bench import corridor_sequence
    clouds, _ = corridor_sequence(ilsm.synth, 14, 0x5EED0100, 40.0)
    for use in (None, [k % 5 != 3 for k in range(len(clouds))]):
        ua = [True if use is None else use[k] for k in range(len(clouds))]
        a = ilsm.Slam(ctx, 0.4, 0.8, 0.3, 4096)
        b = ilsm.Slam(ctx, 0.4, 0.8, 0.3, 4096, pipelined=True)
        sync = [a.frame(c, use_aloam=ua[k]) for k, c in enumerate(clouds)]
        mapped = []
        for k, c in enumerate(clouds):
            qo, to, qm, tm, st = b.frame_async(c, use_aloam=ua[k])
            assert np.array_equal(qo, sync[k][0]) and np.array_equal(to, sync[k][1])
            assert st.ran_odometry == sync[k][4].ran_odometry
            assert (qm is None) == (k == 0)
            if qm is not None:
                mapped.append((qm, tm, st.mapping.pass_[1].num_plane_factors))
        qm, tm, st = b.flush()
        mapped.append((qm, tm, st.mapping.pass_[1].num_plane_factors))
        assert b.flush()[0] is None
        assert len(mapped) == len(clouds)
        for k in range(len(clouds)):
            assert np.array_equal(mapped[k][0], sync[k][2]) and np.array_equal(mapped[k][1], sync[k][3]), k
            assert mapped[k][2] == sync[k][4].mapping.pass_[1].num_plane_factors
        with pytest.raises(ilsm.IlsmError):
            b.frame(clouds[0])
        with pytest.raises(ilsm.IlsmError):
            a.frame_async(clouds[0])
        a.close(), b.close()


def test_cube_merge_voxelgrid_is_bit_identical_to_the_general_pass(ctx, ilsm, monkeypatch):
    """The per-frame VoxelGrid of a map cube merges the new points into the previous pass's output (ilsm_voxel.cuh
    voxelgrid_block_merge) and skips cubes nothing was inserted into; ILSM_VG_MERGE=0 sends every pass through the
    general hash / sort VoxelGrid instead.  Poses and every cube of both maps must agree bit for bit."""
    import torch
    S = ilsm.synth
    frames = 160
    scene = S.Scene(corridor=True, length=0.2 * frames + 30.0)
    clouds = S.make_frames_torch(scene, S.corridor_poses(frames), 0x5EED0120, torch.device("cuda:0"))
    clouds = [clouds[k].numpy() for k in range(frames)]
    runs = []
    for flag in ("1", "0"):
        monkeypatch.setenv("ILSM_VG_MERGE", flag)
        slam = ilsm.Slam(ctx, 0.4, 0.8, 0.3, 8192)
        poses = [slam.frame(c)[2:4] for c in clouds]
        cm = slam.cubemap()
        cubes = {}
        for which in (0, 1):
            for idx in range(21 * 21 * 11):
                pts = cm.cube(which, idx)
                if len(pts):
                    cubes[(which, idx)] = pts.copy()
        runs.append((poses, cubes))
        slam.close()
    (pa, ca), (pb, cb) = runs
    for k in range(len(clouds)):
        assert np.array_equal(pa[k][0], pb[k][0]) and np.array_equal(pa[k][1], pb[k][1]), k
    assert sorted(ca) == sorted(cb) and len(ca) > 4
    assert max(len(v) for v in ca.values()) > 2048, max(len(v) for v in ca.values())  # the large-cube path is exercised
    for key in ca:
        assert ca[key].tobytes() == cb[key].tobytes(), key


def _run_staged(slam, clouds, use_aloam=None):
    """Push every cloud through ilsm_slam_frame_staged, then drain; returns ({frame: (q, t)} odometry, {frame: ...} mapped,
    {frame: stats of the call that returned its odometry})."""
    odom, mapped, stats = {}, {}, {}
    seq = list(clouds) + [None, None]
    for k, c in enumerate(seq):
        ua = True if (use_aloam is None or c is None) else use_aloam[k]
        fo, qo, to, fm, qm, tm, st = slam.frame_staged(c, use_aloam=ua)
        assert fo == (k - 1 if 1 <= k <= len(clouds) else -1), (k, fo)
        assert fm == (k - 2 if 2 <= k <= len(clouds) + 1 else -1), (k, fm)
        if fo >= 0:
            odom[fo] = (qo, to)
            stats[fo] = st
        if fm >= 0:
            mapped[fm] = (qm, tm, st.mapping.pass_[1].num_plane_factors)
    fo, _, _, fm, _, _, _ = slam.frame_staged(None)  # an empty pipeline stays empty
    assert fo == -1 and fm == -1
    return odom, mapped, stats


def test_three_stage_loop_gives_the_same_poses(ctx, ilsm):
    """ilsm_slam_create_staged: scanRegistration, laserOdometry and laserMapping as three stages with their own contexts
    and host threads (the reference's three nodes).  Odometry poses arrive one call later, mapped poses two calls later,
    both bit-identical to the synchronous loop -- also when some frames skip the odometry solve (use_aloam = 0 travels
    with the frame) and across a second sequence on the same handle kind."""
    import os, sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    from sequence_bench import corridor_sequence
    clouds, _ = corridor_sequence(ilsm.synth, 18, 0x5EED0110, 40.0)
    for use in (None, [k % 5 != 3 for k in range(len(clouds))]):
        a = ilsm.Slam(ctx, 0.4, 0.8, 0.3, 4096)
        b = ilsm.Slam(ctx, 0.4, 0.8, 0.3, 4096, staged=True)
        sync = [a.frame(c, use_aloam=True if use is None else use[k]) for k, c in enumerate(clouds)]
        odom, mapped, stats = _run_staged(b, clouds, use)
        assert sorted(odom) == sorted(mapped) == list(range(len(clouds)))
        for k in range(len(clouds)):
            assert np.array_equal(odom[k][0], sync[k][0]) and np.array_equal(odom[k][1], sync[k][1]), k
            assert np.array_equal(mapped[k][0], sync[k][2]) and np.array_equal(mapped[k][1], sync[k][3]), k
            assert mapped[k][2] == sync[k][4].mapping.pass_[1].num_plane_factors
            assert stats[k].n_less_flat == sync[k][4].n_less_flat and stats[k].ran_odometry == sync[k][4].ran_odometry
        with pytest.raises(ilsm.IlsmError):
            b.frame(clouds[0])
        with pytest.raises(ilsm.IlsmError):
            b.flush()
        with pytest.raises(ilsm.IlsmError):
            a.frame_staged(clouds[0])
        a.close(), b.close()


def test_three_stage_loop_destroyed_with_frames_in_flight(ctx, ilsm):
    """Destroying a staged handle while its stages still hold frames must drain them, not hang or crash."""
    import os, sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    from sequence_bench import corridor_sequence
    clouds, _ = corridor_sequence(ilsm.synth, 4, 0x5EED0111, 40.0)
    b = ilsm.Slam(ctx, 0.4, 0.8, 0.3, 4096, staged=True)
    for c in clouds:
        b.frame_staged(c)
    b.close()


@pytest.mark.parametrize("mode", ["synchronous", "pipelined", "staged"])
def test_feature_clouds_above_16384_points(ctx, oracle_mod, ilsm, mode):
    """A 64-ring sensor whose beams all fall inside the reference's +-22.5 degree ring formula keeps every return
    (scanRegistration.cpp:308-316, 570-589): ~17.7 k less-flat points per frame in the open scene -- more than one block's
    VoxelGrid sorts.  The full loop routes such clouds through the tiled multi-block VoxelGrid and must still match the
    chained oracle, in the synchronous loop, with the mapping stage pipelined and as three stages."""
    S = ilsm.synth
    scene = S.Scene()
    q0, t0 = S.default_pose()
    frames = []
    for k in range(4):
        q = S.quat_mul(q0, S.quat_from_rotvec([0.0, 0.0, 0.01 * k]))
        t = np.asarray(t0) + [0.15 * k, 0.02 * k, 0.0]
        frames.append(S.make_frame(scene, q, t, seed=0x5EED0700 + k, fov_deg=22.0)[0])
    slam = ilsm.Slam(ctx, 0.4, 0.8, 0.3, 16384, pipelined=mode == "pipelined", staged=mode == "staged")
    oslam = oracle_mod.Slam(0.4, 0.8, 0.3)
    want = [oslam.frame(cloud) for cloud in frames]
    if mode == "staged":
        _, mapped, st = _run_staged(slam, frames)
        got, stats = [mapped[k][:2] for k in range(len(frames))], [st[k] for k in range(len(frames))]
    elif mode == "pipelined":
        got, stats = [], []
        for cloud in frames:
            qo, to, qm, tm, st = slam.frame_async(cloud)
            stats.append(st)
            if qm is not None:
                got.append((qm, tm))
        got.append(slam.flush()[:2])
    else:
        runs = [slam.frame(cloud) for cloud in frames]
        got, stats = [r[2:4] for r in runs], [r[4] for r in runs]
    assert len(got) == len(want)
    for k, ((gq, gt), (_, w, info), st) in enumerate(zip(got, want, stats)):
        assert st.n_less_flat == len(info["features"]["less_flat"]) and st.n_less_flat > 16384, (k, st.n_less_flat)
        assert st.n_less_sharp == len(info["features"]["less_sharp_idx"])
        assert np.linalg.norm(gt - w[4:]) < 1e-4 and S.quat_angle(gq, w[:4]) < 1e-4, k
    slam.close()


def test_long_run_with_in_loop_window_rolls_matches_oracle(ctx, oracle_mod, ilsm):
    """laserMapping's 21x21x11 window of 50 m cubes rolls when the centre cube comes within 3 cubes of the border
    (laserMapping.cpp:341-565): 0.6 m per frame along a 460 m corridor crosses that line twice inside the loop (at ~375 m
    and ~425 m of estimated travel).  Every pose, the window indices and the whole occupied map must match the chained oracle."""
    import torch
    S = ilsm.synth
    F = 760
    scene = S.Scene(corridor=True, length=0.6 * F + 30.0)
    poses = S.corridor_poses(F, step=0.6)
    clouds = S.make_frames_torch(scene, poses, 0x5EED0900, torch.device("cuda:0"))
    slam = ilsm.Slam(ctx, 0.4, 0.8, 0.3, 8192)
    oslam = oracle_mod.Slam(0.4, 0.8, 0.3)
    cen, ocen = [], []
    for k in range(F):
        cloud = clouds[k].numpy()
        gqo, gto, gqm, gtm, st = slam.frame(cloud)
        wodom, wmap, info = oslam.frame(cloud)
        assert np.linalg.norm(gtm - wmap[4:]) < 1e-4 and S.quat_angle(gqm, wmap[:4]) < 1e-4, k
        assert np.linalg.norm(gto - wodom[4:]) < 1e-4, k
        assert st.cubemap.flags == 0
        cen.append(tuple(st.cubemap.cen))
        ocen.append(tuple(info["cubemap"].cen))
    rolls = [k for k in range(1, F) if cen[k] != cen[k - 1]]
    assert cen == ocen and len(rolls) >= 2, rolls
    view = slam.cubemap()
    occupied = [i for i in range(4851) if len(oslam.cube.cube(1, i)) or len(oslam.cube.cube(0, i))]
    assert len(occupied) >= 8
    for idx in occupied:
        for which in (0, 1):
            g, w = view.cube(which, idx), oslam.cube.cube(which, idx)
            assert g.shape == w.shape and np.array_equal(g[:, :3], w[:, :3]), (idx, which)
    slam.close()


def test_cube_capacity_overflow_is_reported(ctx, ilsm):
    """A cube slab that cannot take the frame's points must not corrupt anything silently: the frame call fails with
    ILSM_ERR_OUT_OF_MEMORY and names the capacity flag (32 = cube slab full)."""
    S = ilsm.synth
    frames = corridor_frames(S, 6)
    slam = ilsm.Slam(ctx, 0.4, 0.8, 0.3, 512)  # 512 points per 50 m cube: the first frames already overflow it
    with pytest.raises(ilsm.IlsmError) as ei:
        for cloud, _, _ in frames:
            slam.frame(cloud)
    assert ei.value.code == -5 and "capacity" in str(ei.value) and "0x2" in str(ei.value)
    slam.close()
