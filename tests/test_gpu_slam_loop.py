"""Loop closure as a stage of the full loop (ilsm_slam_enable_loop) on the GPU, over the closed-loop sequence of
synth.closed_loop_poses(): equal byte for byte to the composition of a handle without loop closure, the keyframe rule
restated in Python, ctx.extract_features' cloud and an ilsm_loop on a second context; the same across the synchronous,
pipelined and three-stage loops; poses untouched; revisits accepted near the truth; back-pressure; the results API;
teardown with keyframes in flight; launch counts."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
MODES = ("sync", "pipelined", "staged")
OPTS_A = dict(exclude_recent=20, tree_period=1, sc_dist_threshold=0.3)  # the revisit option set
MIN_RANGE = 0.3
# the box scene's edges at 0.4 m fill a 50 m cube beyond its 16384 points: map the less-sharp cloud at 0.6 m
LINE_RES = 0.6


@pytest.fixture(scope="module")
def seq(ilsm):
    import torch
    S = ilsm.synth
    poses = S.closed_loop_poses()
    clouds = S.make_frames_torch(S.Scene(), poses, 0x5EED3000, torch.device("cuda:0"))
    return poses, [clouds[k].numpy() for k in range(len(poses))]


def make(ilsm, ctx, mode, loop=None):
    slam = ilsm.Slam(ctx, LINE_RES, 0.8, MIN_RANGE, 16384, pipelined=mode == "pipelined", staged=mode == "staged",
                     mapping="mapOptimization" if mode == "mapopt" else "laserMapping")
    if loop is not None:
        slam.enable_loop(**loop)
    return slam


def drive(slam, mode, clouds):
    """Every frame through the handle; returns ({frame: (q_odom, t_odom)}, {frame: (q_map, t_map)})."""
    odom, mapped = {}, {}
    if mode in ("sync", "mapopt"):
        for k, c in enumerate(clouds):
            qo, to, qm, tm, _ = slam.frame(c)
            odom[k], mapped[k] = (qo, to), (qm, tm)
    elif mode == "pipelined":
        for k, c in enumerate(clouds):
            qo, to, qm, tm, _ = slam.frame_async(c)
            odom[k] = (qo, to)
            if qm is not None:
                mapped[k - 1] = (qm, tm)
        qm, tm, _ = slam.flush()
        mapped[len(clouds) - 1] = (qm, tm)
    else:
        for k in range(len(clouds) + 2):
            fo, qo, to, fm, qm, tm, _ = slam.frame_staged(clouds[k] if k < len(clouds) else None)
            if fo >= 0:
                odom[fo] = (qo, to)
            if fm >= 0:
                mapped[fm] = (qm, tm)
    assert sorted(mapped) == list(range(len(clouds))) and sorted(odom) == list(range(len(clouds)))
    return odom, mapped


def run(ilsm, ctx, mode, clouds, loop=None):
    slam = make(ilsm, ctx, mode, loop)
    odom, mapped = drive(slam, mode, clouds)
    events = slam.loop_results(wait=True) if loop is not None else None
    slam.close()
    return odom, mapped, events


def compose(ilsm, ctx, clouds, mapped, keyframe_dist=1.0, keyframe_angle_rad=0.2, max_pending=8, **loop_opts):
    """The same decisions from the existing entry points: the mapped poses of a handle without loop closure, the keyframe
    rule restated, the front end's cloud from ctx.extract_features and an ilsm_loop on a context of its own."""
    S = ilsm.synth
    poses = [mapped[k] for k in range(len(clouds))]
    kfs = S.select_keyframes(poses, keyframe_dist, keyframe_angle_rad)
    c2 = ilsm.Context(0)
    lc = ilsm.LoopClosure(c2, **loop_opts)
    out = []
    for k in kfs:
        cloud = ctx.extract_features(clouds[k], MIN_RANGE)["cloud"]
        out.append((k, poses[k], bytes(lc.add_keyframe(cloud, *poses[k]))))
    lc.close(), c2.close()
    return out


def same_events(events, composed):
    assert [e.frame for e in events] == [k for k, _, _ in composed]
    for i, (e, (k, (q, t), r)) in enumerate(zip(events, composed)):
        assert e.result.keyframe_id == i
        assert e.q.tobytes() == np.asarray(q, np.float64).tobytes() and e.tv.tobytes() == np.asarray(t, np.float64).tobytes(), k
        assert bytes(e.result) == r, (i, k)


def event_bytes(events):
    return [bytes(e) for e in events]


@pytest.fixture(scope="module")
def runs(ilsm, ctx, seq):
    """Each cube-map mode over the whole sequence with loop closure off and on (option set A)."""
    _, clouds = seq
    return {(mode, on): run(ilsm, ctx, mode, clouds, OPTS_A if on else None) for mode in MODES for on in (False, True)}


def test_equals_the_composition_byte_for_byte(ilsm, ctx, seq, runs):
    _, clouds = seq
    _, mapped, events = runs[("sync", True)]
    composed = compose(ilsm, ctx, clouds, runs[("sync", False)][1], **OPTS_A)
    same_events(events, composed)
    assert 60 < len(events) < 140 and any(e.result.verified for e in events)


def test_every_frame_a_keyframe_at_the_defaults(ilsm, ctx, seq):
    _, clouds = seq
    clouds = clouds[:72]
    opts = dict(keyframe_dist=0.0, keyframe_angle_rad=0.0)
    _, plain, _ = run(ilsm, ctx, "sync", clouds)
    _, _, events = run(ilsm, ctx, "sync", clouds, opts)
    assert len(events) == len(clouds)
    same_events(events, compose(ilsm, ctx, clouds, plain, **opts))
    assert all(e.result.nn_id == -1 for e in events[:50]) and all(e.result.nn_id >= 0 for e in events[50:])


def test_the_same_across_modes(runs):
    want = event_bytes(runs[("sync", True)][2])
    for mode in ("pipelined", "staged"):
        assert event_bytes(runs[(mode, True)][2]) == want, mode


def test_mapoptimization_handle_equals_its_composition(ilsm, ctx, seq):
    _, clouds = seq
    clouds = clouds[:90]
    opts = dict(exclude_recent=5, tree_period=1, sc_dist_threshold=0.3)
    _, plain, _ = run(ilsm, ctx, "mapopt", clouds)
    _, mapped, events = run(ilsm, ctx, "mapopt", clouds, opts)
    for k in range(len(clouds)):
        assert mapped[k][0].tobytes() == plain[k][0].tobytes() and mapped[k][1].tobytes() == plain[k][1].tobytes(), k
    same_events(events, compose(ilsm, ctx, clouds, plain, **opts))
    assert len(events) > 10


@pytest.mark.parametrize("mode", MODES)
def test_poses_are_unchanged(runs, mode):
    (o0, m0, _), (o1, m1, _) = runs[(mode, False)], runs[(mode, True)]
    for k in o0:
        for a, b in zip(o0[k] + m0[k], o1[k] + m1[k]):
            assert a.tobytes() == b.tobytes(), (mode, k)
    # and the three modes agree with each other, as without loop closure
    s = runs[("sync", True)][1]
    assert all(m1[k][1].tobytes() == s[k][1].tobytes() for k in m1)


def test_revisits_found_and_wrong_places_rejected(ilsm, seq, runs):
    """Every accepted loop joins two views of the same place, and the second lap's revisits of the first are accepted.
    The rotation of T_loop^-1 * T_icp is within 0.5 degrees of the true relative pose for every accepted loop.  Its
    translation is within 5 cm (median) for revisits 0.1 m from the stored keyframe, the setting of test_gpu_loop.py's
    bar; further apart, the ICP's early stop (transformation_epsilon) leaves it short of the truth by up to about a
    quarter of the offset: 2-6 cm at 0.1 m, 5-12 cm at 0.27 m, 10-13 cm at 0.52 m on this sequence."""
    S = ilsm.synth
    poses, _ = seq
    events = runs[("sync", True)][2]
    n_lap = len(poses) // 2
    accepted = [e for e in events if e.result.accepted]
    errors = {}
    for e in accepted:
        k, c = int(e.frame), int(events[e.result.loop_id].frame)
        (qk, tk), (qc, tc) = poses[k], poses[c]
        qi = S.quat_inv(qc)
        q_rel, t_rel = S.quat_mul(qi, qk), S.quat_to_mat(qi) @ (tk - tc)
        errors[k] = (c, float(np.linalg.norm(tk - tc)), float(np.linalg.norm(e.result.tv - t_rel)),
                     float(np.rad2deg(S.quat_angle(e.result.q, q_rel))))
        print(f"frame {k} -> frame {c}: {errors[k][1]:.2f} m apart, sc {e.result.sc_dist:.3f}, fitness {e.result.icp.fitness:.4f}, "
              f"error {100 * errors[k][2]:.2f} cm / {errors[k][3]:.3f} deg")
    print(f"{len(events)} keyframes, {sum(e.result.verified for e in events)} verified, {len(accepted)} accepted")
    assert all(d < 3.0 for _, d, _, _ in errors.values()), errors  # no loop with another place
    revisits = {k: v for k, v in errors.items() if k >= n_lap and v[0] < n_lap}
    assert revisits, [(e.frame, e.result.loop_id, e.result.sc_dist) for e in events if e.result.verified]
    assert all(ea < 0.5 and et < 0.05 + 0.3 * d for _, d, et, ea in errors.values()), errors
    near = [et for _, d, et, _ in revisits.values() if d < 0.15]
    assert len(near) >= 10 and np.median(near) < 0.05, near


def test_back_pressure_keeps_the_order(ilsm, ctx, seq, runs):
    """max_pending = 1 with three-stage frames pushed back to back: every keyframe waits for the previous answer."""
    _, clouds = seq
    _, _, events = run(ilsm, ctx, "staged", clouds, dict(OPTS_A, max_pending=1))
    assert event_bytes(events) == event_bytes(runs[("sync", True)][2])


def test_results_api(ilsm, ctx, seq):
    _, clouds = seq
    n = 30
    slam = make(ilsm, ctx, "sync", dict(keyframe_dist=0.0, keyframe_angle_rad=0.0, exclude_recent=5, tree_period=1))
    got = []
    for k in range(n):
        slam.frame(clouds[k])
        part = slam.loop_results(wait=False)  # answered ones only, in order
        assert [e.frame for e in part] == list(range(len(got), len(got) + len(part)))
        got += part
    first = slam.loop_results(wait=True, capacity=3)
    assert [e.frame for e in first] == list(range(len(got), len(got) + min(3, n - len(got))))
    got += first
    rest = slam.loop_results(wait=False)  # everything is answered after the wait: the rest is ready
    got += rest
    assert [e.frame for e in got] == list(range(n)) and [e.result.keyframe_id for e in got] == list(range(n))
    assert slam.loop_results(wait=True) == [] and slam.loop_results(wait=False, capacity=0) == []
    with pytest.raises(ilsm.IlsmError) as ei:  # after the first frame
        slam.enable_loop()
    assert ei.value.code == -6
    slam.close()
    plain = make(ilsm, ctx, "sync")
    with pytest.raises(ilsm.IlsmError) as ei:  # not on
        plain.loop_results()
    assert ei.value.code == -6
    plain.enable_loop()
    with pytest.raises(ilsm.IlsmError) as ei:  # already on
        plain.enable_loop()
    assert ei.value.code == -6
    plain.close()


@pytest.mark.parametrize("mode", MODES + ("mapopt",))
def test_destroyed_with_keyframes_in_flight(ilsm, seq, mode):
    _, clouds = seq
    before = ilsm.live_bytes()
    c = ilsm.Context(0)
    slam = make(ilsm, c, mode, dict(keyframe_dist=0.0, keyframe_angle_rad=0.0, exclude_recent=3, tree_period=1, max_pending=4,
                                    sc_dist_threshold=1.0))
    for k in range(12):
        if mode == "staged":
            slam.frame_staged(clouds[k])
        elif mode == "pipelined":
            slam.frame_async(clouds[k])
        else:
            slam.frame(clouds[k])
    slam.close()
    c.close()
    assert ilsm.live_bytes() == before


def test_no_launches_for_frames_that_are_not_keyframes(ilsm, ctx, seq):
    """The synchronous loop, where every launch of a frame happens inside its call: the same count per frame without loop
    closure and with it on for a frame that is not a keyframe."""
    _, clouds = seq
    lc = ilsm.launch_count
    a = make(ilsm, ctx, "sync")
    b = make(ilsm, ctx, "sync", dict(keyframe_dist=1e9, keyframe_angle_rad=1e9))  # frame 0 only
    counts = []
    for k in range(12):
        per = []
        for s in (a, b):
            b0 = lc()
            s.frame(clouds[k])
            per.append(lc() - b0)
        if k == 0:  # the one keyframe: let its answer come before counting on
            assert len(b.loop_results(wait=True)) == 1
        counts.append(per)
    for k in range(1, 12):
        assert counts[k][0] == counts[k][1], (k, counts)
    a.close(), b.close()
