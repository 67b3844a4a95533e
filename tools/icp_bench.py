"""Loop-closure verification throughput: ilsm_icp_align_batch on the box-scene loop workload.

Workload (synth.loop_keyframes): keyframes of a closed two-lap path through synth.Scene(); source = one OS0-64 frame after
VoxelGrid(0.4) in the sensor frame; target = world-frame submap of +-2 keyframes around a ScanContext candidate of the
first lap, VoxelGrid(0.4), in an ilsm_map with a 1 m cell; guess = the candidate's pose turned by the ScanContext shift
(6 degrees per sector).  Batches of 1 (the best candidate of one query), 10 (one query's candidates) and 148 (every
query's candidates, repeated).  Reports pairs/s timed with CUDA events on the library's stream (warm-up, then at least
1 s of calls), iterations per pair, launches per call, the oracle's single-thread time for the batch-1 pair, and the
device name and power limit read in the same run.  Writes icp_bench.json under --out."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

OPTS = dict(max_correspondence_distance=2.0, max_iterations=50, transformation_epsilon=1e-8, euclidean_fitness_epsilon=1e-6)


def device_info():
    import torch
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        info["nvidia_smi"] = r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unavailable"
    except (OSError, subprocess.SubprocessError):
        info["nvidia_smi"] = "unavailable"
    return info


def workload(ilsm, ctx, n_per_lap=12):
    import numpy as np
    S = ilsm.synth
    kfs = S.loop_keyframes(n_per_lap=n_per_lap)
    db = ilsm.ScanContextDb(ctx)
    db.add(np.stack([db.make_scancontext(k["src"]) for k in kfs[:n_per_lap]]))
    submaps = [S.loop_submap(kfs, c, n_per_lap) for c in range(n_per_lap)]
    maps = [ctx.new_map().set_input_cloud(m, 1.0) for m in submaps]
    queries = []  # per query: [(candidate, source, guess)] in candidate order
    for k in kfs[n_per_lap:]:
        ids, _, dist, shifts = db.query_candidates(db.make_scancontext(k["src"]), num_candidates=10)
        order = np.argsort(np.where(ids >= 0, dist, np.inf), kind="stable")
        pairs = []
        for i in order:
            if ids[i] < 0:
                continue
            c = int(ids[i])
            q0 = S.quat_mul(kfs[c]["q"], S.quat_from_rotvec([0.0, 0.0, np.deg2rad(6.0 * int(shifts[i]))]))
            pairs.append((c, k["src"], (q0, kfs[c]["t"])))
        queries.append(pairs)
    db.close()
    return kfs, submaps, maps, queries


def time_batch(ilsm, ctx, maps, pairs, min_s=1.0):
    import torch
    targets, sources, guesses = [maps[c] for c, _, _ in pairs], [s for _, s, _ in pairs], [g for _, _, g in pairs]
    for _ in range(3):
        res = ctx.icp_align_batch(targets, sources, guesses, **OPTS)
    before = ilsm.launch_count()
    ctx.icp_align_batch(targets, sources, guesses, **OPTS)
    launches = ilsm.launch_count() - before
    stream = torch.cuda.ExternalStream(ctx.stream_ptr)
    calls, dev_s, t0 = 0, 0.0, time.perf_counter()
    while time.perf_counter() - t0 < min_s:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(5):
            ctx.icp_align_batch(targets, sources, guesses, **OPTS)
        b.record(stream)
        b.synchronize()
        dev_s += a.elapsed_time(b) / 1e3
        calls += 5
    its = [r.iterations for r in res]
    return {"pairs": len(pairs), "calls": calls, "device_s": dev_s, "pairs_per_s": calls * len(pairs) / dev_s,
            "ms_per_call": 1e3 * dev_s / calls, "iterations_mean": float(sum(its)) / len(its), "iterations_max": max(its),
            "launches_per_call": launches, "accepted": sum(1 for r in res if r.converged and r.fitness < 0.3)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", required=True, help="output directory (icp_bench.json)")
    ap.add_argument("--min-seconds", type=float, default=1.0)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("icp_bench: no CUDA device (this measurement has no CPU fallback)")
    import ilsm_b200 as ilsm
    from oracle import icp as oracle_icp
    ctx = ilsm.Context(0)
    kfs, submaps, maps, queries = workload(ilsm, ctx)
    all_pairs = [p for q in queries for p in q]
    batches = {"1": queries[0][:1], "10": queries[0][:10], "148": [all_pairs[i % len(all_pairs)] for i in range(148)]}
    out = {"workload": "synth.loop_keyframes(12 per lap, 2 laps), VoxelGrid(0.4), submap +-2 keyframes, cell 1 m",
           "opts": OPTS, "source_points_mean": float(sum(len(s) for _, s, _ in all_pairs)) / len(all_pairs),
           "target_points_mean": float(sum(len(m) for m in submaps)) / len(submaps), **device_info(), "batches": {}}
    for name, pairs in batches.items():
        out["batches"][name] = time_batch(ilsm, ctx, maps, pairs, args.min_seconds)
        print(name, out["batches"][name], flush=True)
    c, src, (q0, t0) = batches["1"][0]
    reps, t_or = 0, time.perf_counter()
    while reps < 3 or time.perf_counter() - t_or < 1.0:
        w = oracle_icp.icp_align(submaps[c], src, q0, t0, **OPTS)
        reps += 1
    out["oracle_single_thread_s_per_pair"] = (time.perf_counter() - t_or) / reps
    out["oracle_note"] = "the oracle's 1-NN entry point rebuilds its k-d tree of the target on every iteration"
    out["oracle_iterations"] = w.iterations
    for m in maps:
        m.close()
    ctx.close()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "icp_bench.json"), "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
