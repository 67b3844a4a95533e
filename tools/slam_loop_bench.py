"""Loop closure as a stage of the full loop (ilsm_slam_enable_loop): what it costs the frame rate, and how fast keyframes
are answered.  One process, loop closure off and on alternated (off, on, on, off) on the same frames:

  corridor   the 2000-frame corridor of config 2 (bench.py) through the three-stage and the synchronous loop, default
             loop options (keyframe every 1 m / 0.2 rad, exclude_recent 50).  The path never comes back, but the corridor
             repeats itself every 5 m, so ScanContext finds "loops" and the ICP verifies (and accepts) many of them: the
             keyframes, verified and accepted loops are recorded with the rates.
  closed     the two-lap closed-loop sequence of synth.closed_loop_poses() (exclude_recent 20, tree period 1, threshold
             0.3; line resolution 0.6 m, cube capacity 16384).

Per run: frames/s over the frame calls (the ilsm_slam_loop_results polls of the "on" runs are timed apart and left out),
the host phases of ilsm_slam_host_phases, the ILSM_STAGE_TRACE lines, and with loop closure the latency of each keyframe
from the call that selects it to the first ilsm_slam_loop_results(wait = 0) poll that returns it (polled after every call,
so the resolution is one call).  Then the same keyframes -- the front end's cloud of each keyframe frame, its mapped pose
-- through a standalone ilsm_loop (ilsm_loop_add_keyframe_dev, clouds already on the device) on the otherwise idle GPU,
one call at a time with a host clock around each: the loop stage's work without the full loop beside it, by kind (early
return, searched without a loop, verified).

The card's name and power limit are read in the same run.  Writes slam_loop_bench.json under --out (default profiles/)."""
from __future__ import annotations

import argparse
import json
import os
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(ROOT))
sys.path.insert(0, ROOT)

LOOP_CLOSED = dict(exclude_recent=20, tree_period=1, sc_dist_threshold=0.3)
CLOSED_MAP = (0.6, 16384)  # line resolution and cube capacity of the closed loop: the box scene's edges fill a cube at 0.4 m


def traced_close(slam):
    """Destroy the handle with its ILSM_STAGE_TRACE lines (written to fd 2) captured."""
    with tempfile.TemporaryFile(mode="w+") as tf:
        sys.stderr.flush()
        saved = os.dup(2)
        os.dup2(tf.fileno(), 2)
        try:
            slam.close()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
        tf.seek(0)
        return [line.strip() for line in tf if "stage trace" in line]


def replay(ilsm, ctx, views, mode, loop, line_res=0.4, cube_capacity=8192):
    """All frames through one handle; returns the run's numbers and, with loop closure, its events and latencies."""
    slam = ilsm.Slam(ctx, line_res, 0.8, 0.3, cube_capacity, staged=mode == "staged")
    if loop is not None:
        slam.enable_loop(**loop)
    ctx.sync()
    F = len(views)
    lag = 2 if mode == "staged" else 0  # the call that hands out frame f's mapped pose is call f + lag
    handed, latency, events = {}, [], []
    t0 = time.perf_counter()
    poll = 0.0  # time in the loop_results polls, left out of the frame rate
    for k in range(F + lag):
        if mode == "staged":
            slam.frame_staged(views[k] if k < F else None)
        else:
            slam.frame(views[k])
        if loop is not None:
            now = time.perf_counter()
            if k - lag >= 0:
                handed[k - lag] = now
            for e in slam.loop_results(wait=False):
                latency.append(now - handed[int(e.frame)])
                events.append(e)
            poll += time.perf_counter() - now
    wall = time.perf_counter() - t0 - poll
    if loop is not None:
        tw = time.perf_counter()
        rest = slam.loop_results(wait=True)
        latency += [tw - handed[int(e.frame)] for e in rest]
        events += rest
    phases = slam.host_phases()
    trace = traced_close(slam)
    out = {"frames_per_s": round(F / wall, 1), "ms_per_frame": round(1e3 * wall / F, 4), "wall_s": round(wall, 4),
           "poll_ms_per_frame": round(1e3 * poll / F, 4),
           "host_phase_ms_per_frame": [round(1e3 * float(p) / F, 4) for p in phases], "stage_trace": trace}
    return out, events, latency


def standalone(ilsm, ctx, views, events, opts):
    """The keyframes of `events` through a standalone ilsm_loop on a context of its own, device input, one timed call each."""
    import numpy as np
    import torch
    clouds = [torch.from_numpy(np.ascontiguousarray(ctx.extract_features(views[int(e.frame)], 0.3)["cloud"])).cuda() for e in events]
    torch.cuda.synchronize()
    c2 = ilsm.Context(0)
    lc = ilsm.LoopClosure(c2, **opts)
    kinds = {"early_return": [], "searched_no_loop": [], "verified": []}
    same = True
    for e, cl in zip(events, clouds):
        t0 = time.perf_counter()
        r = lc.add_keyframe_dev(cl, e.q, e.tv)
        dt = time.perf_counter() - t0
        same = same and bytes(r) == bytes(e.result)
        kinds["verified" if r.verified else "early_return" if r.nn_id < 0 else "searched_no_loop"].append(dt)
    lc.close(), c2.close()
    out = {k: {"calls": len(v), "median_ms": pct(v, 50), "p90_ms": pct(v, 90), "total_s": round(float(np.sum(v)), 4)}
           for k, v in kinds.items()}
    out["total_s"] = round(float(sum(np.sum(v) for v in kinds.values())), 4)
    out["identical_results"] = bool(same)
    return out


def pct(a, q):
    import numpy as np
    return round(1e3 * float(np.percentile(a, q)), 3) if len(a) else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=2000)
    ap.add_argument("--out", default=os.path.join(os.path.dirname(ROOT), "profiles"))
    a = ap.parse_args()
    os.environ["ILSM_STAGE_TRACE"] = "1"
    import numpy as np
    import torch
    import ilsm_b200 as ilsm
    from loop_bench import device_info
    S = ilsm.synth
    dev = torch.device("cuda:0")
    ctx = ilsm.Context(0)
    result = {"device": device_info(), "order": "per mode: loop closure off, on, on, off"}
    # corridor of config 2 (the frames bench.py replays)
    scene = S.Scene(corridor=True, length=0.2 * a.frames + 30.0)
    clouds = S.make_frames_torch(scene, S.corridor_poses(a.frames), 0x5EED0100, dev)
    views = [clouds[k].numpy() for k in range(a.frames)]
    for mode in ("staged", "sync"):
        replay(ilsm, ctx, views[:100], mode, {})  # warm-up: both contexts' allocations, the loop stage's first keyframes
        runs = {"off": [], "on": []}
        kf = None
        for on in (False, True, True, False):
            r, ev, lat = replay(ilsm, ctx, views, mode, {} if on else None)
            if on:
                kf, kf_events = len(ev), ev
                r["keyframes"], r["verified"] = len(ev), sum(int(e.result.verified) for e in ev)
                r["accepted"] = sum(int(e.result.accepted) for e in ev)
                r["latency_ms_median"], r["latency_ms_p90"] = pct(lat, 50), pct(lat, 90)
            runs["on" if on else "off"].append(r)
        fps = {k: [x["frames_per_s"] for x in v] for k, v in runs.items()}
        result[f"corridor_{mode}"] = {"frames": a.frames, "keyframes": kf, "runs": runs,
                                      "loop_stage_alone": standalone(ilsm, ctx, views, kf_events, {}),
                                      "frames_per_s_mean": {k: round(float(np.mean(v)), 1) for k, v in fps.items()},
                                      "change_pct": round(100.0 * (np.mean(fps["on"]) / np.mean(fps["off"]) - 1.0), 2)}
    del clouds, views
    # closed-loop sequence
    poses = S.closed_loop_poses()
    clouds = S.make_frames_torch(S.Scene(), poses, 0x5EED3000, dev)
    views = [clouds[k].numpy() for k in range(len(poses))]
    for mode in ("staged", "sync"):
        replay(ilsm, ctx, views[:100], mode, LOOP_CLOSED, *CLOSED_MAP)
        runs = {"off": [], "on": []}
        for on in (False, True, True, False):
            r, ev, lat = replay(ilsm, ctx, views, mode, LOOP_CLOSED if on else None, *CLOSED_MAP)
            if on:
                kf_events = ev
                r["keyframes"] = len(ev)
                r["verified"] = sum(int(e.result.verified) for e in ev)
                r["accepted"] = sum(int(e.result.accepted) for e in ev)
                r["accepted_later_lap"] = sum(int(e.result.accepted and e.frame >= len(poses) // 2) for e in ev)
                r["latency_ms_median"], r["latency_ms_p90"] = pct(lat, 50), pct(lat, 90)
            runs["on" if on else "off"].append(r)
        fps = {k: [x["frames_per_s"] for x in v] for k, v in runs.items()}
        result[f"closed_loop_{mode}"] = {"frames": len(poses), "options": LOOP_CLOSED, "runs": runs,
                                         "loop_stage_alone": standalone(ilsm, ctx, views, kf_events, LOOP_CLOSED),
                                         "frames_per_s_mean": {k: round(float(np.mean(v)), 1) for k, v in fps.items()}}
    result["device_after"] = device_info()
    ctx.close()
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "slam_loop_bench.json"), "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps({k: (v.get("frames_per_s_mean"), v.get("change_pct")) for k, v in result.items() if isinstance(v, dict) and "runs" in v}))


if __name__ == "__main__":
    main()
