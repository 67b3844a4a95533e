"""Closing a handle frees every device and pinned byte and every CUDA event, stream and graph exec it allocated.  The
library counts the bytes its buffers hold (ilsm_debug_live_bytes) and the CUDA handles its owners hold
(ilsm_debug_live_handles); cudaMemGetInfo cannot show this on a GPU that other processes use too."""
import gc
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_nothing_is_held_before_a_context_exists(ilsm):
    """A fresh process, so that no other test has created a context yet; reading the count makes no CUDA call."""
    r = subprocess.run([sys.executable, "-c", "import ilsm_b200; print(*ilsm_b200.live_bytes(), ilsm_b200.live_handles())"],
                       cwd=ROOT, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert r.stdout.split() == ["0", "0", "0"]


def corridor_frames(S, n_frames, seed0=0x5EED0A00):
    scene = S.Scene(corridor=True, length=120.0)
    out = []
    for k in range(n_frames):
        q = S.quat_from_rotvec([0.0, 0.0, np.deg2rad(5.0) * np.sin(2 * np.pi * k / 50.0)])
        t = np.array([2.0 + 0.2 * k, 0.1 * np.sin(k / 15.0), 1.2])
        out.append(S.make_frame(scene, q, t, seed=seed0 + k)[0])
    return out


def live(ilsm):
    return ilsm.live_bytes() + (ilsm.live_handles(),)


def exercise_every_handle(ilsm, frames, kfs):
    """Open a fresh context, run every kind of handle on it, close everything; returns the live bytes and handles seen
    while open."""
    S = ilsm.synth
    ctx = ilsm.Context(0)
    # LocalMap: build, k-NN (enough queries for the binned path and its query map), Add_Points
    c = S.config1(n_map=20_000)
    m = ctx.new_map().set_input_cloud(c["map_surf"])
    rng = np.random.default_rng(1)
    qs = (c["map_surf"][rng.integers(0, len(c["map_surf"]), 10_000)] + rng.normal(0, 0.2, (10_000, 3))).astype(np.float32)
    m.nearest_k_search(qs, 5)
    m.add_points(c["map_corner"])
    # ScanContext database: the second add outgrows the first reservation (descriptors and ring keys are copied over)
    db = S.sc_database(600)
    q, _, _ = S.sc_queries(db, 4)
    sc = ilsm.ScanContextDb(ctx)
    sc.add(db[:100])
    sc.add(db[100:])
    sc.query_topk_batch(q, k=10)
    sc.prefilter_debug(q)
    # cube map, ground extraction, mapOptimization
    f = ctx.extract_features(frames[0])
    cm = ilsm.CubeMap(ctx, 0.4, 0.8)
    cm.frame(f["cloud"][f["less_sharp_idx"]], f["less_flat"], [0, 0, 0, 1], [0, 0, 0])
    ge = ilsm.GroundExtractor(ctx)
    ge.extract(frames[0])
    mo = ilsm.MapOptimization(ctx)
    for k in range(2):
        fk = ctx.extract_features(frames[k])
        mo.frame(frames[k], fk["less_flat"], [0, 0, 0, 1], [0.2 * k, 0, 0])
    # loop closure per keyframe
    lc = ilsm.LoopClosure(ctx, tree_period=1)
    for kf in kfs:
        lc.add_keyframe(kf["src"], kf["q"], kf["t"])
    # the full loop in all four modes, with loop closure on: every frame a keyframe, none of their answers collected
    slams = [ilsm.Slam(ctx, 0.4, 0.8, 0.3, 4096), ilsm.Slam(ctx, mapping="mapOptimization"),
             ilsm.Slam(ctx, 0.4, 0.8, 0.3, 4096, pipelined=True), ilsm.Slam(ctx, 0.4, 0.8, 0.3, 4096, staged=True)]
    for s in slams:
        s.enable_loop(keyframe_dist=0.0, keyframe_angle_rad=0.0, max_pending=4, exclude_recent=3, tree_period=1)
    # a refused enable_loop (after the first frame) creates nothing
    plain = ilsm.Slam(ctx, 0.4, 0.8, 0.3, 4096)
    plain.frame(frames[0])
    before = live(ilsm)
    with pytest.raises(ilsm.IlsmError) as ei:
        plain.enable_loop()
    assert ei.value.code == -6
    assert live(ilsm) == before
    for cloud in frames:
        slams[0].frame(cloud)
        slams[1].frame(cloud)
        slams[2].frame_async(cloud)
        slams[3].frame_staged(cloud)
    slams[2].flush()
    for _ in range(2):  # the staged loop's last two frames are still being mapped
        slams[3].frame_staged(None)
    held = live(ilsm)
    for h in slams + [plain, lc, mo, ge, cm, sc, m]:
        h.close()
    ctx.close()
    return held


@pytest.mark.gpu
def test_closing_every_handle_returns_to_the_baseline(ilsm):
    frames = corridor_frames(ilsm.synth, 6)
    kfs = ilsm.synth.loop_keyframes(n_per_lap=4, laps=1)
    gc.collect()  # handles that earlier tests left to the garbage collector must not close during the cycles
    base = live(ilsm)
    for cycle in range(2):
        held = exercise_every_handle(ilsm, frames, kfs)
        assert all(h > b for h, b in zip(held, base)), (cycle, held, base)
        assert live(ilsm) == base, cycle
