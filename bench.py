#!/usr/bin/env python
"""bench.py -- scan-to-map registrations/s on B200 (BASELINE.json metric), one JSON line on stdout.

A "step" is one pass of the reference's per-frame mapping hot section over one synthetic OS0-64 frame
(laserMapping.cpp:624-861): rebuild the corner and surf search structures over the 100k-point local map
(kdtree->setInputCloud x2), then 2 x [associate every stack point (pose transform, exact 5-NN, line/plane fit)
+ ceres::Solve (LM, <= 4 iterations)].

  value : device-timed (CUDA events on the library's stream), map + feature stacks already resident in HBM.
  e2e   : the same step through the host-pointer C ABI (ilsm_map_build x2 + ilsm_register) from pinned host
          buffers, host<->device copies inside the timed region, wall-clocked around the blocking calls;
          median over >= 200 repetitions (p90 alongside).
  roofline     : the step's kernels timed alone (solve, associate, map build), the dominant one as `roofline`,
                 algorithmic bytes / time.
  cpu_baseline : the CPU restatement of the reference path (single thread like the reference's mapping thread) on a
                 bounded sample of the same workload -- on the reference's own nanoflann k-d tree when oracle/_ref
                 holds it; `cpu_baselines` adds the k-NN-only (all cores), front-end and ikd-Tree baselines.

Sub-records (other BASELINE.json configs, measured in the same run):
  config1_with_frontend  N = 1   the frame through front end -> stacks -> registration (ilsm_register_frame)
  config2                N = 1   configs[1]: the full odometry + mapping loop over a 2000-frame corridor sequence,
                                 every pose compared with the chained CPU oracle (window rolls included)
  config3                N = 1   configs[2]: k-NN (exact and gated) and J^T J kernels at N = 2 M / Q = 65 536 / 4 M factors
  config4                any N   configs[3]: independent sequences over the N GPUs (weak: one per GPU; strong: 8 in all)
  config5                any N   configs[4]: ScanContext scoring over a 100k-keyframe database sharded N ways, one NCCL
                                 all-gather of the per-rank top-k per query batch behind the C ABI

`--impl reference` times the CPU path alone (the reference itself cannot be built here, see DESIGN.md).
`--dump-outputs DIR` writes the pose the last timed step computed to DIR/pose.npy (both arms; the inputs are seeded).
N > 1 (torchrun): the headline is independent replicas, one per GPU, no data-path collective ("scaling": "weak").
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "scan-to-map registrations/sec (OS0-64 frame, 100k-pt map)"
UNIT = "registrations/s"
N_MAP = 100_000
SEQ_SEED = 0x5EED0100


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------------------------------------------
# clocks, affinity, L2
# ----------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons of ONE GPU sampled every 50 ms through NVML while the timed regions run (rank 0
    only: one in-process thread instead of an nvidia-smi child per rank)."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, torch, cuda_index):
        self.sm, self.mx, self.reasons = [], [], set()
        self.stop_flag = threading.Event()
        self.thread = None
        self.err = None
        try:
            import pynvml
            pynvml.nvmlInit()
            pr = torch.cuda.get_device_properties(cuda_index)
            bus = "%08x:%02x:%02x.0" % (getattr(pr, "pci_domain_id", 0), pr.pci_bus_id, pr.pci_device_id)
            try:
                self.h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(cuda_index)
            self.nv = pynvml
        except Exception as e:  # NVML missing: report it, the run itself is unaffected
            self.nv, self.err = None, repr(e)

    def _loop(self):
        nv = self.nv
        while not self.stop_flag.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                self.mx.append(float(nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)))
                get = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
                mask = int(get(self.h))
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception as e:
                self.err = repr(e)
            self.stop_flag.wait(0.05)

    def start(self):
        if self.nv is not None:
            self.thread = threading.Thread(target=self._loop, daemon=True)
            self.thread.start()
        return self

    def stop(self):
        self.stop_flag.set()
        if self.thread is not None:
            self.thread.join(timeout=2)
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: " + str(self.err)], "samples": 0}
        return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": max(self.mx), "reasons": sorted(self.reasons),
                "samples": len(self.sm), "source": "nvml, 50 ms period, rank 0"}


def pin_affinity(torch, local_rank, world):
    """Every rank on its own slice of the host cores, taken from the cores NVML names as local to its GPU when that is
    known (the ranks that share a NUMA node split it), else an even split of the allowed set."""
    try:
        allowed = sorted(os.sched_getaffinity(0))
        groups = None
        try:
            import pynvml
            pynvml.nvmlInit()
            words = (max(allowed) // 64) + 1
            ideal = []
            for r in range(world):
                pr = torch.cuda.get_device_properties(r)
                bus = "%08x:%02x:%02x.0" % (getattr(pr, "pci_domain_id", 0), pr.pci_bus_id, pr.pci_device_id)
                h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
                mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
                cores = [64 * w + b for w in range(words) for b in range(64) if (int(mask[w]) >> b) & 1]
                ideal.append(tuple(c for c in cores if c in allowed))
            groups = ideal
        except Exception:
            groups = None
        if groups and groups[local_rank]:
            mine = groups[local_rank]
            peers = [r for r in range(world) if groups[r] == mine]
            per = max(1, len(mine) // len(peers))
            k = peers.index(local_rank)
            cores = list(mine[k * per:(k + 1) * per]) or list(mine)
        else:
            per = max(1, len(allowed) // world)
            cores = allowed[local_rank * per:(local_rank + 1) * per] or allowed
        os.sched_setaffinity(0, cores)
        return len(cores)
    except Exception:
        return None


class L2Flush:
    """Cold L2 between timed iterations: write a 256 MiB buffer (> the 126 MB L2), then read a second 256 MiB buffer so
    that the lines left in L2 are CLEAN -- otherwise the timed kernel pays for the write-back of ~100 MB of dirty flush
    lines, which is not its traffic."""

    def __init__(self, torch, dev):
        self.w = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        self.r = torch.zeros(64 << 20, dtype=torch.float32, device=dev)  # float: one reduce kernel, no widening copy
        self.sink = None

    def zero_(self):
        self.w.zero_()
        self.sink = self.r.sum()


def workload(seed_shift=0):
    import ilsm_b200 as ilsm
    return ilsm.synth.config1(n_map=N_MAP, seed_shift=seed_shift)


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the step's kernels, from the committed ncu --set full
    capture of this workload (newest profiles/r0N_ncu_traffic.json; empty when absent)."""
    for name in ("r02_ncu_traffic.json", "r01_ncu_traffic.json"):
        try:
            return json.load(open(os.path.join(ROOT, "profiles", name)))
        except Exception:
            continue
    return {}


def pad4(a):
    out = np.zeros((len(a), 4), np.float32)
    out[:, :3] = a[:, :3]
    return out


# ----------------------------------------------------------------------------------------------------
# config 3: bandwidth regime of the two hot kernels
# ----------------------------------------------------------------------------------------------------
def config3_point(ilsm, torch, ctx, ext, flush, dev, peak, opts):
    """BASELINE configs[2], largest point of tools/sweep.py: exact 5-NN of a whole 65536-point frame in a 2M-point map
    (exact: max_dist 0; gated: max_dist 1.0 m = the reference's d2[4] < 1.0 acceptance radius, results beyond it are
    "don't care"), and the J^T J kernel on 4M factors (64 frames' worth in one launch)."""
    S = ilsm.synth
    c = S.config1(n_map=2_000_000)
    m = np.zeros((len(c["map_corner"]) + len(c["map_surf"]), 4), np.float32)
    m[:, :3] = np.concatenate([c["map_corner"], c["map_surf"]])[:, :3]
    d_m = torch.from_numpy(m).to(dev)
    R = S.quat_to_mat(c["q_true"])
    w = np.zeros((65536, 4), np.float32)
    w[:, :3] = (c["cloud"][:, :3].astype(np.float64) @ R.T + c["t_true"]).astype(np.float32)
    d_q = torch.from_numpy(w).to(dev)
    d_idx = torch.empty((65536, 5), dtype=torch.int32, device=dev)
    d_d2 = torch.empty((65536, 5), dtype=torch.float32, device=dev)
    out = {}
    traffic = ncu_traffic().get("config3", {})

    def timed(fn, reps=10):
        ts = []
        with torch.cuda.stream(ext):
            for _ in range(3):
                fn()
            ctx.sync()
            for _ in range(reps):
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(ext)
                fn()
                e1.record(ext)
                ctx.sync()
                ts.append(e0.elapsed_time(e1))
        return float(np.median(ts))

    gm = ctx.new_map()
    with torch.cuda.stream(ext):
        gm.build_dev(d_m.data_ptr(), len(m), 16)
    byt = 16 * len(m) + 56 * 65536
    touched = traffic.get("knn_binned_kernel")
    for tag, md in (("knn5_exact", 0.0), ("knn5_gated", 1.0)):
        t = timed(lambda: gm.knn_dev(d_q.data_ptr(), 65536, 16, 5, md, d_idx.data_ptr(), d_d2.data_ptr()))
        out[tag] = {"N": len(m), "Q": 65536, "max_dist": md, "ms": t, "queries_per_s": 65536 / t * 1e3, "algorithmic_bytes": byt,
                    "achieved_GBs": byt / t / 1e6, "frac": byt / t / 1e6 / peak,
                    "ncu_dram_bytes": touched, "frac_of_bytes_touched": (touched / t / 1e6 / peak) if touched else None,
                    "path": "query binning (count / alloc / scatter over the query cloud + work list) + knn_binned_kernel",
                    "bound": "instruction issue / L2 latency: the queries visit their 27 voxels, not the whole map, so 16 N "
                             "overstates the bytes an exact search has to touch"}
    # J^T J: 4M factors produced by associating 64 copies of the frame against the same map
    hc, hs = pad4(c["map_corner"]), pad4(c["map_surf"])
    d_mc, d_ms = torch.from_numpy(hc).to(dev), torch.from_numpy(hs).to(dev)
    mc, ms = ctx.new_map(), ctx.new_map()
    Qb = 1 << 22
    sens = np.zeros((Qb, 4), np.float32)
    sens[:, :3] = c["cloud"][np.arange(Qb) % 65536, :3]
    d_c, d_s = torch.from_numpy(sens[:Qb // 8].copy()).to(dev), torch.from_numpy(sens[Qb // 8:].copy()).to(dev)
    pose_t = torch.from_numpy(np.concatenate([c["q_true"], c["t_true"]])).to(dev)
    out32 = torch.zeros(32, dtype=torch.float64, device=dev)
    with torch.cuda.stream(ext):
        mc.build_dev(d_mc.data_ptr(), len(hc), 16)
        ms.build_dev(d_ms.data_ptr(), len(hs), 16)
        ctx.associate_dev(mc, ms, d_c.data_ptr(), Qb // 8, d_s.data_ptr(), Qb - Qb // 8, 16, pose_t.data_ptr(), opts)
        ctx.sync()
    t_as = timed(lambda: ctx.associate_dev(mc, ms, d_c.data_ptr(), Qb // 8, d_s.data_ptr(), Qb - Qb // 8, 16, pose_t.data_ptr(), opts), reps=5)
    out["associate"] = {"points": Qb, "corner": Qb // 8, "kernel": "associate_kernel (transform + exact 5-NN + line / plane fit per point)",
                        "ms": t_as, "points_per_s": Qb / t_as * 1e3}
    t = timed(lambda: ctx.eval_normal_eq_dev(pose_t.data_ptr(), out32.data_ptr()))
    # every factor slot read once: type 4 B + point 16 B + (normal | point_a) 32 B, + point_b 32 B for the corner slots
    byt = Qb * 52 + (Qb // 8) * 32
    out["jtj"] = {"factors": Qb, "corner_slots": Qb // 8, "kernel": "normal_eq_bulk_kernel",
                  "ncu_dram_bytes": traffic.get("normal_eq_bulk_kernel"), "ms": t, "factors_per_s": Qb / t * 1e3,
                  "algorithmic_bytes": byt, "achieved_GBs": byt / t / 1e6, "frac": byt / t / 1e6 / peak, "bound": "hbm"}
    gm.close(), mc.close(), ms.close()
    return out


# ----------------------------------------------------------------------------------------------------
# config 1 with its front end
# ----------------------------------------------------------------------------------------------------
def config1_frontend_point(ilsm, torch, ctx, ext, flush, dev, c, mc, ms, d_mc, d_ms, h_mc, h_ms, opts, use_cpu):
    """SURVEY 8d config 1 as the reference pipeline runs it: organised frame -> laserCloudHandler -> less-sharp / less-flat
    clouds -> VoxelGrid(0.4 / 0.8) -> 2 x (associate + LM <= 4) against the 100k map, map structures rebuilt every step."""
    frame = np.ascontiguousarray(c["cloud"][:, :4], np.float32)
    p_frame = torch.from_numpy(frame).pin_memory()
    d_frame = p_frame.to(dev)
    pose0 = np.concatenate([c["q0"], c["t0"]])
    d_pose0 = torch.from_numpy(pose0).to(dev)
    d_pose = d_pose0.clone()

    def step_dev():
        d_pose.copy_(d_pose0, non_blocking=True)
        mc.build_pair_dev(d_mc.data_ptr(), len(h_mc), ms, d_ms.data_ptr(), len(h_ms), 16)
        ctx.register_frame_dev(mc, ms, d_frame.data_ptr(), len(frame), 16, d_pose.data_ptr(), 0.3, 0.4, 0.8, opts)

    ts = []
    with torch.cuda.stream(ext):
        for _ in range(5):
            step_dev()
        ctx.sync()
        for _ in range(30):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(ext)
            step_dev()
            e1.record(ext)
            ctx.sync()
            ts.append(e0.elapsed_time(e1))
    pose = d_pose.cpu().numpy()
    # host-pointer path: frame and both maps from pinned host memory
    p_mc, p_ms = torch.from_numpy(h_mc).pin_memory(), torch.from_numpy(h_ms).pin_memory()
    n_mc, n_ms, n_fr = p_mc.numpy(), p_ms.numpy(), p_frame.numpy()
    ctx.set_async(True)
    es = []
    for k in range(40):
        t0 = time.perf_counter()
        mc.set_input_cloud(n_mc), ms.set_input_cloud(n_ms)
        q, t, rep, sizes = ctx.register_frame(mc, ms, n_fr, c["q0"], c["t0"], 0.3, 0.4, 0.8, opts)
        if k >= 5:
            es.append(time.perf_counter() - t0)
    ctx.set_async(False)
    out = {"workload": "configs[0] with its front end: organised 64x1024 frame -> laserCloudHandler -> VoxelGrid(0.4 / 0.8) stacks "
                       "-> 2 x voxel-hash build + 2 x (associate + LM<=4) vs the 100k map (ilsm_register_frame)",
           "value": 1e3 / float(np.median(ts)), "unit": UNIT, "ms_per_step": float(np.median(ts)),
           "timing": "CUDA events on the library stream around the step (one host synchronisation inside: the feature counts)",
           "e2e": {"value": 1.0 / float(np.median(es)), "unit": UNIT, "ms_per_step": 1e3 * float(np.median(es)),
                   "ms_per_step_p90": 1e3 * float(np.percentile(es, 90)),
                   "h2d_bytes_per_step": int(frame.nbytes + h_mc.nbytes + h_ms.nbytes + 56), "d2h_bytes_per_step": 56 + 8 + 8 * 48 + 40},
           "sizes": {"n_less_sharp": sizes[0], "n_less_flat": sizes[1], "n_corner_stack": sizes[2], "n_surf_stack": sizes[3]},
           "pose_error_m": float(np.linalg.norm(pose[4:] - c["t_true"]))}
    if use_cpu:
        import oracle
        t0 = time.perf_counter()
        f = oracle.extract_features(frame)
        t_fe = time.perf_counter() - t0
        sc_ = oracle.voxelgrid(f["cloud"][f["less_sharp_idx"]], 0.4)
        ss_ = oracle.voxelgrid(f["less_flat"], 0.8)
        x, _, _ = oracle.register_aloam(c["map_corner"], c["map_surf"], sc_, ss_, pose0)
        out["vs_oracle"] = {"pose_diff_m": float(np.linalg.norm(t - x[4:])), "pose_diff_rad": float(ilsm.synth.quat_angle(q, x[:4])),
                            "stack_sizes_equal": bool((len(sc_), len(ss_)) == (sizes[2], sizes[3]))}
        out["cpu_frontend_ms"] = 1e3 * t_fe
    return out


# ----------------------------------------------------------------------------------------------------
# config 2: the full loop over a long sequence
# ----------------------------------------------------------------------------------------------------
def make_sequence(ilsm, torch, dev, frames, seed):
    S = ilsm.synth
    scene = S.Scene(corridor=True, length=0.2 * frames + 30.0)
    poses = S.corridor_poses(frames)
    clouds = S.make_frames_torch(scene, poses, seed, dev)  # pinned (F, 65536, 4) float32
    return clouds, poses


def config2_point(ilsm, torch, ctx, dev, frames, oracle_frames):
    """BASELINE configs[1]: the full per-frame loop (scanRegistration -> laserOdometry -> laserMapping) on a synthetic
    OS0-64 corridor sequence through ilsm_slam_frame (H2D of the organised frame and D2H of both poses inside the timed
    region), the chained CPU oracle over the same frames, and the pose difference frame by frame -- including the frames
    after the 21x21x11 cube window has rolled (the centre cube comes within 3 cubes of the border after ~375 m)."""
    S = ilsm.synth
    t0 = time.perf_counter()
    clouds, poses = make_sequence(ilsm, torch, dev, frames, SEQ_SEED)
    gen_s = time.perf_counter() - t0
    views = [clouds[k].numpy() for k in range(frames)]
    warm = ilsm.Slam(ctx, 0.4, 0.8, 0.3, 8192)
    for k in range(min(5, frames)):
        warm.frame(views[k])
    warm.close()
    slam = ilsm.Slam(ctx, 0.4, 0.8, 0.3, 8192)
    ctx.sync()
    l0 = ilsm.launch_count()
    est, times, cen, flags = [], [], [], 0
    for k in range(frames):
        t0 = time.perf_counter()
        qo, to, qm, tm, st = slam.frame(views[k])
        times.append(time.perf_counter() - t0)
        est.append((qm, tm))
        cen.append(tuple(st.cubemap.cen))
        flags |= int(st.cubemap.flags)
    launches = ilsm.launch_count() - l0
    slam.close()
    wall = float(np.sum(times))
    rolls = [k for k in range(1, frames) if cen[k] != cen[k - 1]]
    q0, t0p = poses[0]
    R0 = S.quat_to_mat(q0)
    err = [float(np.linalg.norm(est[k][1] - R0.T @ (poses[k][1] - t0p))) for k in range(frames)]
    out = {"workload": f"configs[1]: {frames}-frame synthetic OS0-64 corridor ({0.2 * frames:.0f} m), full odometry + mapping loop per frame",
           "value": frames / wall, "unit": "frames/s", "ms_per_frame": 1e3 * wall / frames,
           "ms_per_frame_median": 1e3 * float(np.median(times)), "h2d_bytes_per_frame": int(views[0].nbytes),
           "d2h_bytes_per_frame": 2 * 56 + 400, "gpu_launches_per_frame": launches / frames,
           "ate_rmse_m": float(np.sqrt(np.mean(np.square(err)))), "final_position_error_m": err[-1],
           "window_rolls_in_loop": len(rolls), "first_roll_frame": rolls[0] if rolls else None, "capacity_flags": flags,
           "slowest_frames_ms": {int(k): round(1e3 * times[k], 3) for k in np.argsort(times)[-5:][::-1]},
           "frames_over_1ms": int(np.sum(np.array(times) > 1e-3)),
           "frame_generation_s": gen_s,
           "timing": "host wall clock around the blocking ilsm_slam_frame calls"}
    # the same sequence with laserMapping as its own pipeline stage (ilsm_slam_create_async: second context + host thread,
    # frame k's mapping overlaps frame k+1's front end and odometry; mapped poses arrive one call later, bit-identical)
    wall_p, mapped = None, None
    for _ in range(2):  # first pass warms the second context's allocations
        pslam = ilsm.Slam(ctx, 0.4, 0.8, 0.3, 8192, pipelined=True)
        n_p = frames if _ else min(frames, 100)
        mapped, t0 = [], time.perf_counter()
        for k in range(n_p):
            r = pslam.frame_async(views[k])
            if r[2] is not None:
                mapped.append(r[3])
        mapped.append(pslam.flush()[1])
        wall_p = time.perf_counter() - t0
        pslam.close()
    out["pipelined_mapping_stage"] = {"value": frames / wall_p, "unit": "frames/s", "ms_per_frame": 1e3 * wall_p / frames,
                                      "identical_to_synchronous": bool(all(np.array_equal(a, b[1]) for a, b in zip(mapped, est))),
                                      "note": "mapped pose of frame k returned by call k+1 (one-frame latency, like the "
                                              "reference's separate laserMapping node)"}
    # ... and as three stages (ilsm_slam_create_staged: front end, odometry and mapping each on its own context and host
    # thread, like the reference's three nodes; odometry pose one call later, mapped pose two calls later)
    wall_s, smapped, sodom = None, None, None
    for _ in range(2):
        sslam = ilsm.Slam(ctx, 0.4, 0.8, 0.3, 8192, staged=True)
        n_s = frames if _ else min(frames, 100)
        smapped, sodom, t0 = {}, {}, time.perf_counter()
        stimes, tp = [], t0
        for k in range(n_s + 2):
            fo, qo, to, fm, qm, tm, st = sslam.frame_staged(views[k] if k < n_s else None)
            if fo >= 0:
                sodom[fo] = to
            if fm >= 0:
                smapped[fm] = tm
            tn = time.perf_counter()
            stimes.append(tn - tp)
            tp = tn
        wall_s = time.perf_counter() - t0
        phases = sslam.host_phases()
        sslam.close()
    out["three_stage_pipeline"] = {"value": frames / wall_s, "unit": "frames/s", "ms_per_frame": 1e3 * wall_s / frames,
                                   "identical_to_synchronous": bool(len(smapped) == frames and all(np.array_equal(smapped[k], est[k][1]) for k in range(frames))),
                                   "host_phase_ms_per_frame": [round(1e3 * float(p) / frames, 4) for p in phases],
                                   "ms_per_call_median": 1e3 * float(np.median(stimes)),
                                   "slowest_calls_ms": {int(k): round(1e3 * stimes[k], 3) for k in np.argsort(stimes)[-5:][::-1]},
                                   "note": "odometry pose of frame k returned by call k+1, mapped pose by call k+2 (the "
                                           "reference's three nodes have the same queue latency between them)"}
    no = min(oracle_frames, frames)
    if no > 0:
        import oracle
        osl = oracle.Slam(0.4, 0.8, 0.3)
        t1 = time.perf_counter()
        ores = [osl.frame(views[k]) for k in range(no)]
        cpu_wall = time.perf_counter() - t1
        dm = np.array([float(np.linalg.norm(est[k][1] - ores[k][1][4:])) for k in range(no)])
        dr = np.array([float(S.quat_angle(est[k][0], ores[k][1][:4])) for k in range(no)])
        after = [k for k in range(no) if rolls and k >= rolls[0]]
        out["cpu_baseline"] = {"value": no / cpu_wall, "unit": "frames/s", "cores": 1, "kind": "port",
                               "sample": f"the first {no} frames of the same sequence through the chained CPU oracle"}
        out["max_pose_diff_vs_oracle"] = {"m": float(dm.max()), "rad": float(dr.max()), "frames": no,
                                          "m_after_first_roll": float(dm[after].max()) if after else None,
                                          "frames_after_first_roll": len(after)}
    return out, clouds, poses


# ----------------------------------------------------------------------------------------------------
# config 4: independent sequences over the GPUs
# ----------------------------------------------------------------------------------------------------
def replay_concurrent(ilsm, device_index, seqs):
    """Replay len(seqs) sequences concurrently on one GPU: one context / stream / host thread each (ctypes releases the
    GIL inside the blocking C call).  Returns (wall seconds, final mapped translation per sequence)."""
    ctxs = [ilsm.Context(device_index) for _ in seqs]
    slams = [ilsm.Slam(c, 0.4, 0.8, 0.3, 8192) for c in ctxs]
    for sl, sq in zip(slams, seqs):
        for k in range(min(3, len(sq))):
            sl.frame(sq[k])
    slams = [(sl.close(), ilsm.Slam(c, 0.4, 0.8, 0.3, 8192))[1] for sl, c in zip(slams, ctxs)]
    last = [None] * len(seqs)

    def run(i):
        for v in seqs[i]:
            last[i] = slams[i].frame(v)[3]

    threads = [threading.Thread(target=run, args=(i,)) for i in range(len(seqs))]
    return ctxs, slams, threads, last


def config4_point(ilsm, torch, dist, dev, local_rank, rank, world, frames, barrier):
    """BASELINE configs[3]: independent synthetic sequences replayed in parallel, no data-path collective.
    weak: one sequence per GPU (N sequences in all); strong: 8 sequences in all, 8 / N per GPU run concurrently."""
    S = ilsm.synth
    total_strong = 8
    mine = [s for s in range(total_strong) if s % world == rank]
    seqs = {}
    for s in mine:
        clouds, _ = make_sequence(ilsm, torch, dev, frames, SEQ_SEED + 4096 * (s + 1))
        seqs[s] = [clouds[k].numpy() for k in range(frames)]
    out = {}
    for tag, ids in (("weak", mine[:1]), ("strong", mine)):
        ctxs, slams, threads, last = replay_concurrent(ilsm, local_rank, [seqs[s] for s in ids])
        barrier()
        t0 = time.perf_counter()
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        el = time.perf_counter() - t0
        barrier()
        tt = torch.tensor([el], dtype=torch.float64, device=dev)
        if dist is not None:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        el_max = float(tt.cpu())
        n_seq = world if tag == "weak" else total_strong
        out[tag] = {"sequences": n_seq, "sequences_per_gpu": len(ids), "frames_per_sequence": frames,
                    "value": n_seq * frames / el_max, "unit": "frames/s", "seconds": el_max}
        for sl, c in zip(slams, ctxs):
            sl.close(), c.close()
    out["workload"] = (f"configs[3]: independent {frames}-frame corridor sequences (seeds differ), full loop per frame, "
                       f"one context / stream / host thread per sequence; no collective")
    out["timing"] = "host wall clock, barrier on both sides, max over ranks"
    return out


# ----------------------------------------------------------------------------------------------------
# config 5: sharded ScanContext scoring
# ----------------------------------------------------------------------------------------------------
def config5_point(ilsm, torch, dist, ctx, ext, dev, rank, world, n_kf, n_q, batch, peak, barrier):
    """BASELINE configs[4]: a 100k-keyframe ScanContext database split into contiguous id ranges, one per rank; per
    query batch every rank scores its shard, the packed per-rank top-k records are exchanged with ONE ncclAllGather and
    merged by the same kernel on every rank -- all behind the C ABI (ilsm_sc_init_nccl_rank + ilsm_sc_query_topk_sharded_dev)."""
    S = ilsm.synth
    K = 10
    lo, hi = ilsm.shard_range(n_kf, rank, world)
    sc = ilsm.ScanContextDb(ctx)
    for a in range(lo, hi, 20000):
        sc.add(S.sc_database_range(a, min(hi, a + 20000), n_kf))
    assert len(sc) == hi - lo
    q, ids, shifts = S.sc_chunked_queries(n_kf, n_q)
    d_q = torch.from_numpy(q.reshape(n_q, 1200)).to(dev)
    n_search = max(0, min(hi, n_kf - 50) - lo)  # NUM_EXCLUDE_RECENT: the newest 50 keyframes are never candidates
    if world > 1:
        uid = [ilsm.ScanContextDb.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        sc.init_nccl_rank(uid[0], world, rank)
    merged = torch.zeros((n_q, 16 * K), dtype=torch.uint8, device=dev)

    def run_all():
        for b0 in range(0, n_q, batch):
            nb = min(batch, n_q - b0)
            sc.query_topk_sharded_dev(d_q[b0].data_ptr(), nb, K, n_search, lo, merged[b0].data_ptr())

    with torch.cuda.stream(ext):
        sc.query_topk_sharded_dev(d_q[0].data_ptr(), min(batch, n_q), K, n_search, lo, merged[0].data_ptr())
        ctx.sync()
        barrier()
        l0 = ilsm.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(ext)
        run_all()
        e1.record(ext)
        ctx.sync()
        barrier()
        launches = ilsm.launch_count() - l0
        ms = e0.elapsed_time(e1)
    tt = torch.tensor([ms], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms = float(tt.cpu())
    m = merged.cpu().numpy()
    top_id = np.array([m[j, 8 * K:12 * K].view(np.int32)[0] for j in range(n_q)])
    top_sh = np.array([m[j, 12 * K:16 * K].view(np.int32)[0] for j in range(n_q)])
    hit = float(np.mean((top_id == ids) & (top_sh == shifts)))
    # reference-exact search on the unsharded database: detectLoopClosureID's 10 ring-key candidates
    cand = None
    if world == 1:
        nq2 = min(n_q, 100)
        t0 = time.perf_counter()
        ok = 0
        for j in range(nq2):
            loop, dmin, sh, nn = sc.detect_loop_closure_id(q[j], n_search)
            ok += int(nn == ids[j] and sh == shifts[j])
        cand = {"queries": nq2, "value": nq2 / (time.perf_counter() - t0), "unit": "queries/s", "top1_id_and_shift_recovered": ok / nq2,
                "what": "ilsm_sc_query_candidates (ring-key 10-NN + 10 distanceBtnScanContext) = SCManager::detectLoopClosureID, "
                        "host call with H2D of the query and D2H of the candidates inside"}
    byt = (n_kf - 50) * 4800.0
    out = {"workload": f"configs[4]: {n_kf} keyframes sharded over {world} rank(s), {n_q} queries in batches of {batch}, top-{K}",
           "value": n_q / ms * 1e3, "unit": "queries/s", "ms_per_query": ms / n_q, "scaling": "strong",
           "db_bytes_per_query": byt, "GBs_aggregate": byt * n_q / ms / 1e6, "frac_of_hbm_peak_x_n": byt * n_q / ms / 1e6 / (peak * world),
           "exchange": (f"one ncclAllGather of {batch} x {16 * K} B per rank per batch (communicator behind the C ABI, "
                        f"NCCL {ilsm.ScanContextDb.nccl_version()})") if world > 1 else "none (1 rank)",
           "gpu_launches": int(launches), "top1_id_and_shift_recovered": hit,
           "timing": "CUDA events on the library stream around the whole query loop, barrier on both sides, max over ranks"}
    if cand is not None:
        out["reference_exact_candidates"] = cand
    sc.close()
    return out


# ----------------------------------------------------------------------------------------------------
# CPU arms
# ----------------------------------------------------------------------------------------------------
def cpu_tree():
    import oracle
    return "nanoflann" if oracle.lib_nanoflann() is not None else "own"


def cpu_registrations_per_s(c, budget_s, min_reps=3):
    import oracle
    tree = cpu_tree()
    qt0 = np.concatenate([c["q0"], c["t0"]])
    mc, ms, co, su = c["map_corner"], c["map_surf"], c["corner"], c["surf"]
    oracle.register_aloam(mc, ms, co, su, qt0, tree=tree)  # warm-up
    reps, t0 = 0, time.perf_counter()
    while True:
        oracle.register_aloam(mc, ms, co, su, qt0, tree=tree)
        reps += 1
        el = time.perf_counter() - t0
        if reps >= min_reps and el >= budget_s:
            break
    return reps / el, reps, el, tree


TREE_NOTE = {"nanoflann": "k-d tree = the reference's vendored nanoflann 1.3.2 (include/nanoflann.hpp, oracle/_ref/libref_aloam.so)",
             "own": "k-d tree = the oracle's private tree (oracle/_ref/libref_aloam.so absent)"}


def extra_cpu_baselines(c, budget_s):
    """The other CPU baselines BASELINE.md section 3 names, each on a bounded sample."""
    import oracle
    out = {}
    tree = cpu_tree()
    # B-knn-omp: k-NN only over all host cores (and on one, for the ratio)
    m = np.ascontiguousarray(np.concatenate([c["map_corner"], c["map_surf"]])[:, :3], np.float32)
    R = __import__("ilsm_b200").synth.quat_to_mat(c["q_true"])
    q = (c["cloud"][:, :3].astype(np.float64) @ R.T + c["t_true"]).astype(np.float32)
    q = q[np.any(c["cloud"][:, :3] != 0, axis=1)]
    res = {}
    for name, th in (("all_cores", 0), ("one_core", 1)):
        best = None
        t0 = time.perf_counter()
        while best is None or time.perf_counter() - t0 < budget_s / 4:
            _, _, used, bs, qs = oracle.knn_kdtree_omp(m, q, 5, th, tree)
            best = (used, bs, qs) if best is None or qs < best[2] else best
        res[name] = {"threads": best[0], "build_ms": 1e3 * best[1], "query_ms": 1e3 * best[2], "queries_per_s": len(q) / best[2]}
    out["knn_all_cores"] = {"value": res["all_cores"]["queries_per_s"], "unit": "queries/s", "cores": res["all_cores"]["threads"],
                            "nproc": os.cpu_count(), "kind": "port", "detail": res,
                            "sample": f"exact 5-NN of {len(q)} frame points in the {len(m)}-point config-1 map, std::thread over the "
                                      f"host cores; {TREE_NOTE[tree]}"}
    # B-frontend: projection + feature extraction, one thread
    frame = np.ascontiguousarray(c["cloud"][:, :4], np.float32)
    n, t0 = 0, time.perf_counter()
    while n < 2 or time.perf_counter() - t0 < budget_s / 4:
        oracle.project(frame)
        oracle.extract_features(frame)
        n += 1
    el = time.perf_counter() - t0
    out["frontend"] = {"value": n / el, "unit": "frames/s", "cores": 1, "kind": "port", "ms_per_frame": 1e3 * el / n,
                       "sample": f"{n} x (cloud_handler + laserCloudHandler) of the config-1 frame"}
    # B-ikd: the reference's OWN ikd-Tree (Build + Nearest_Search + Add_Points per frame) when oracle/_ref holds it
    if oracle.ref_ikd() is not None:
        surf_w = (c["surf"][:, :3].astype(np.float64) @ R.T + c["t_true"]).astype(np.float32)
        tb = time.perf_counter()
        t = oracle.RefIkdTree(0.3, 0.6, 0.4).build(c["map_surf"][:, :3])
        build_s = time.perf_counter() - tb
        n, t0 = 0, time.perf_counter()
        while n < 2 or time.perf_counter() - t0 < budget_s / 4:
            t.nearest(surf_w, 5)
            n += 1
        el = time.perf_counter() - t0
        ta = time.perf_counter()
        t.add_points(surf_w, True)
        add_s = time.perf_counter() - ta
        t.close()
        out["ikd_tree"] = {"value": n * len(surf_w) / el, "unit": "queries/s", "cores": 1, "kind": "reference",
                           "build_ms": 1e3 * build_s, "nearest_search_ms_per_frame": 1e3 * el / n, "add_points_ms": 1e3 * add_s,
                           "sample": f"/root/reference/src/ikd-Tree compiled into oracle/_ref/libref_ikd.so: Build({len(c['map_surf'])} pts), "
                                     f"Nearest_Search(k=5) of the {len(surf_w)}-point surf stack, Add_Points(downsample) of it"}
    return out


def run_reference(args, rank, world):
    """The reference arm: a step is ONE registration of the same frame by the CPU path (same definition as the
    GPU arm).  Rank 0 alone runs it."""
    if rank != 0:
        return
    import oracle
    c = workload()
    tree = cpu_tree()
    qt0 = np.concatenate([c["q0"], c["t0"]])
    a = (c["map_corner"], c["map_surf"], c["corner"], c["surf"], qt0)
    for _ in range(max(args.warmup, 1)):
        oracle.register_aloam(*a, tree=tree)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        x, sums, nf = oracle.register_aloam(*a, tree=tree)
    wall = time.perf_counter() - t0
    assert float(np.linalg.norm(x[4:] - c["t_true"])) < 0.05
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, pose=x)
    value = args.steps / wall
    sample = f"{args.steps} registrations of the config-1 frame in {wall:.2f} s"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * wall / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32 k-NN / f64 fit+solve", "data": "synthetic",
        "config": {"workload": "configs[0] shape: one OS0-64 frame (64x1024) vs 100k-pt local map per step: "
                               "2 x k-d tree build + 2 x (5-NN association + LM<=4); CPU restatement of "
                               "laserMapping.cpp:624-861 (the reference itself cannot be built here)",
                   "n_map": N_MAP, "n_corner_stack": int(len(c["corner"])), "n_surf_stack": int(len(c["surf"]))},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": 1, "kind": "port", "sample": sample,
                         "note": "single thread: the reference runs this path on one thread (laserMapping.cpp:1215 "
                                 "mapping_process, Ceres num_threads default 1); " + TREE_NOTE[tree]},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ----------------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------------
def run_gpu(args, rank, world, local_rank):
    import torch
    import ilsm_b200 as ilsm

    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))
    torch.cuda.set_device(local_rank)
    dev = torch.device(f"cuda:{local_rank}")
    cores = pin_affinity(torch, local_rank, world)

    ilsm._build.build()
    c = workload()  # replicas: every rank registers the same frame against its own copy of the map (fixed work per GPU)
    ctx = ilsm.Context(local_rank)
    ext = torch.cuda.ExternalStream(ctx.stream_ptr, device=dev)
    mc, ms = ctx.new_map(), ctx.new_map()
    opts = ilsm.default_opts()

    # ---- device-resident inputs
    h_mc, h_ms = pad4(c["map_corner"]), pad4(c["map_surf"])
    h_c, h_s = pad4(c["corner"]), pad4(c["surf"])
    pose0 = np.concatenate([c["q0"], c["t0"]])
    d_mc, d_ms = torch.from_numpy(h_mc).to(dev), torch.from_numpy(h_ms).to(dev)
    d_c, d_s = torch.from_numpy(h_c).to(dev), torch.from_numpy(h_s).to(dev)
    d_pose0 = torch.from_numpy(pose0).to(dev)
    d_pose = d_pose0.clone()
    flush = L2Flush(torch, dev)
    torch.cuda.synchronize()

    def step_dev():
        d_pose.copy_(d_pose0, non_blocking=True)
        mc.build_pair_dev(d_mc.data_ptr(), len(h_mc), ms, d_ms.data_ptr(), len(h_ms), 16)  # the two setInputCloud lines in one call
        ctx.register_dev(mc, ms, d_c.data_ptr(), len(h_c), d_s.data_ptr(), len(h_s), 16, d_pose.data_ptr(), opts)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.cuda.stream(ext):
        for _ in range(max(args.warmup, 3)):
            flush.zero_()
            step_dev()
        ctx.sync()
        # sanity: the device path must land on the true pose (no work skipped)
        pose = d_pose.cpu().numpy()
        err_t = float(np.linalg.norm(pose[4:] - c["t_true"]))
        assert err_t < 0.05, f"registration did not converge: {err_t} m"

        sampler = ClockSampler(torch, local_rank).start() if rank == 0 else None
        barrier()
        launches0 = ilsm.launch_count()
        evs = []
        for _ in range(args.steps):
            flush.zero_()  # L2 flush between timed iterations (outside the event pair)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(ext)
            step_dev()
            e1.record(ext)
            evs.append((e0, e1))
        ctx.sync()
        barrier()
        launches = ilsm.launch_count() - launches0
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, pose=d_pose.cpu().numpy())
        ms_steps = [a.elapsed_time(b) for a, b in evs]
        dev_ms = float(np.sum(ms_steps))

        # ---- e2e through the host-pointer ABI from pinned buffers
        p_mc, p_ms = torch.from_numpy(h_mc).pin_memory(), torch.from_numpy(h_ms).pin_memory()
        p_c, p_s = torch.from_numpy(h_c).pin_memory(), torch.from_numpy(h_s).pin_memory()
        n_mc, n_ms, n_c, n_s = p_mc.numpy(), p_ms.numpy(), p_c.numpy(), p_s.numpy()

        # the C ABI called directly (ctypes), argument marshalling hoisted out of the loop: what a C++ caller pays
        import ctypes as C
        lib = ilsm.load_library()
        vp = C.c_void_p
        a_mc, a_ms, a_c, a_s = (vp(x.ctypes.data) for x in (n_mc, n_ms, n_c, n_s))
        qq, tt = np.zeros(4), np.zeros(3)
        a_q, a_t = vp(qq.ctypes.data), vp(tt.ctypes.data)
        rep = ilsm.RegReport()
        a_opts, a_rep = C.byref(opts), C.byref(rep)
        len_mc, len_ms, len_c, len_s = len(n_mc), len(n_ms), len(n_c), len(n_s)
        q_init, t_init = np.asarray(c["q0"], np.float64).copy(), np.asarray(c["t0"], np.float64).copy()

        def step_host():
            qq[:] = q_init
            tt[:] = t_init
            rc = lib.ilsm_map_build(mc._h, a_mc, len_mc, 16, 0.0) or lib.ilsm_map_build(ms._h, a_ms, len_ms, 16, 0.0) or \
                lib.ilsm_register(ctx._h, mc._h, ms._h, a_c, len_c, a_s, len_s, 16, a_q, a_t, a_opts, a_rep)
            if rc:
                raise RuntimeError(lib.ilsm_last_error().decode())
            return qq, tt, rep

        ctx.set_async(True)  # the two setInputCloud replacements overlap (see ilsm_set_async in include/ilsm.h)
        for _ in range(5):
            step_host()
        barrier()
        e2e_reps = max(args.steps, 200)
        e2e_times = []
        for _ in range(e2e_reps):
            flush.zero_()
            ctx.sync()
            t0 = time.perf_counter()
            q, t, rep = step_host()
            e2e_times.append(time.perf_counter() - t0)
        barrier()
        ctx.set_async(False)
        e2e_med, e2e_p90, e2e_p10 = float(np.median(e2e_times)), float(np.percentile(e2e_times, 90)), float(np.percentile(e2e_times, 10))
        assert float(np.linalg.norm(t - c["t_true"])) < 0.05
        h2d = h_mc.nbytes + h_ms.nbytes + h_c.nbytes + h_s.nbytes + 56
        d2h = 56 + 8 + 8 * 48

        # ---- the step's kernels timed alone on the library stream (CUDA events, L2 flushed before each batch)
        def timed(fn, reps=20, batches=5):
            ts = []
            for _ in range(batches):
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(ext)
                for _ in range(reps):
                    fn()
                e1.record(ext)
                ctx.sync()
                ts.append(e0.elapsed_time(e1) / reps)
            return float(np.median(ts))

        mc.build_dev(d_mc.data_ptr(), len(h_mc), 16)
        ms.build_dev(d_ms.data_ptr(), len(h_ms), 16)
        assoc_ms = timed(lambda: ctx.associate_dev(mc, ms, d_c.data_ptr(), len(h_c), d_s.data_ptr(), len(h_s), 16,
                                                   d_pose0.data_ptr(), opts))
        # ceres::Solve replacement: factors from the association at the initial guess, LM <= 4 iterations from that guess
        solve_ms = timed(lambda: ctx.solve_dev(d_pose0.data_ptr(), opts.max_num_iterations, opts.huber_a))
        build_ms = timed(lambda: (mc.build_pair_dev(d_mc.data_ptr(), len(h_mc), ms, d_ms.data_ptr(), len(h_ms), 16), mc.join(), ms.join()))
        clocks = sampler.stop() if sampler is not None else None
    # ---- aggregate over ranks (max time)
    t_dev = torch.tensor([dev_ms, e2e_med * 1e3, e2e_p90 * 1e3, e2e_p10 * 1e3], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t_dev, op=dist.ReduceOp.MAX)
    dev_ms_max, e2e_med_ms, e2e_p90_ms, e2e_p10_ms = [float(x) for x in t_dev.cpu()]
    value = world * args.steps / (dev_ms_max * 1e-3)
    e2e_value = world / (e2e_med_ms * 1e-3)

    peak, peak_src = load_peaks()
    nq = len(h_c) + len(h_s)
    n_map = len(h_mc) + len(h_ms)
    step_ms = dev_ms_max / args.steps
    # algorithmic bytes per launch (DESIGN.md section 5): every input read once, every output written once
    assoc_bytes = 16 * n_map + nq * (16 + 84)           # map points + stack point in + factor record out
    solve_bytes = nq * 84 + 1024                        # factor records read once (kept in registers across the LM evaluations)
    build_bytes = 48 * n_map                            # points in, keys/ranks r+w, grouped points out (both maps)
    traffic = ncu_traffic().get("config1", {})
    kernels = []
    for name, ms_k, byt, per_step in (("solve_cluster_kernel", solve_ms, solve_bytes, 2), ("associate_kernel", assoc_ms, assoc_bytes, 2),
                                      ("grid_{count,alloc,scatter}_kernel (both maps, 3 launches)", build_ms, build_bytes, 1)):
        kernels.append({"kernel": name, "launch_ms": ms_k, "launches_per_step": per_step,
                        "share_of_step": per_step * ms_k / step_ms, "algorithmic_bytes": int(byt),
                        "achieved_GBs": byt / (ms_k * 1e-3) / 1e9, "frac": byt / (ms_k * 1e-3) / 1e9 / peak,
                        "ncu_dram_bytes": traffic.get(name.split(" ")[0].split("(")[0])})
    dom = max(kernels[:2], key=lambda k: k["share_of_step"])

    single = rank == 0 and world == 1
    fe_rec = sweep = seq = cpu = cpu_more = None
    if single and not args.no_frontend:
        fe_rec = config1_frontend_point(ilsm, torch, ctx, ext, flush, dev, c, mc, ms, d_mc, d_ms, h_mc, h_ms, opts, not args.no_cpu)
    if single and not args.no_sweep:
        sweep = config3_point(ilsm, torch, ctx, ext, flush, dev, peak, opts)
    if single and not args.no_sequence:
        seq, _, _ = config2_point(ilsm, torch, ctx, dev, args.sequence_frames, 0 if args.no_cpu else args.sequence_oracle_frames)
    c4 = c5 = None
    if not args.no_sharded:
        c4 = config4_point(ilsm, torch, dist, dev, local_rank, rank, world, args.config4_frames, barrier)
        c5 = config5_point(ilsm, torch, dist, ctx, ext, dev, rank, world, args.sc_keyframes, args.sc_queries, args.sc_batch, peak, barrier)
    if single and not args.no_cpu:
        v, reps_cpu, el, tree = cpu_registrations_per_s(c, args.cpu_seconds, 5)
        cpu = {"value": v, "unit": UNIT, "cores": 1, "kind": "port",
               "sample": f"{reps_cpu} registrations of the same frame/map in {el:.1f} s (CPU restatement, 1 thread: the "
                         f"reference's mapping loop is single-threaded, laserMapping.cpp:1215); {TREE_NOTE[tree]}"}
        cpu_more = extra_cpu_baselines(c, args.cpu_seconds)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": dev_ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 k-NN / f64 fit+solve", "data": "synthetic",
            "config": {"workload": "configs[0] shape: one OS0-64 frame (64x1024) vs 100k-pt local map per step: "
                                   "2 x voxel-hash build + 2 x (associate + LM<=4); one independent frame per GPU",
                       "n_map": N_MAP, "n_corner_stack": int(len(h_c)), "n_surf_stack": int(len(h_s)),
                       "l2": "flushed between timed iterations (256 MiB write + 256 MiB read of a second buffer: cold and clean)",
                       "parallelism": f"replicas x{world}", "host_cores_per_rank": cores},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": e2e_med_ms, "ms_per_step_p10": e2e_p10_ms, "ms_per_step_p90": e2e_p90_ms, "reps": e2e_reps,
                    "timing": "host wall clock around the blocking C-ABI calls; median over the repetitions, max over ranks"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": dom["kernel"], "achieved": dom["achieved_GBs"], "peak": peak,
                         "unit": "GB/s", "frac": dom["frac"], "traffic": dom["ncu_dram_bytes"], "peak_source": peak_src,
                         "algorithmic_bytes": dom["algorithmic_bytes"], "kernel_ms": dom["launch_ms"],
                         "kernels": kernels,
                         "note": "config-1 sizes are latency-bound, not bandwidth-bound: one launch moves 0.2-2 MB "
                                 "(0.03-0.3 us at peak) and the LM loop is a serial chain of <= 5 evaluations of dependent "
                                 "fp64 arithmetic (~35 cycles per dependent op) with a cluster exchange each; the shares are "
                                 "of kernels timed ALONE, so they can add up to more than 1 (the two map builds overlap in "
                                 "the step); the bandwidth regime of the same kernels is in `config3` and in profiles/"},
            "clocks": clocks,
            "pose_error_m": err_t,
        }
        for key, val in (("config1_with_frontend", fe_rec), ("config2", seq), ("config3", sweep), ("config4", c4), ("config5", c5),
                         ("cpu_baseline", cpu), ("cpu_baselines", cpu_more)):
            if val is not None:
                line[key] = val
        emit(line)
    mc.close(), ms.close(), ctx.close()
    if dist is not None:
        dist.destroy_process_group()


_RESULT_OUT = None


def claim_stdout():
    """The contract is ONE JSON line on stdout.  Native code prints there too (the NCCL banner; the reference's ikd-Tree,
    timed as a CPU baseline, announces its rebuild thread with printf), so file descriptor 1 is pointed at stderr for the
    whole run and the result line goes to a private duplicate of the original stdout."""
    global _RESULT_OUT
    if _RESULT_OUT is None:
        sys.stdout.flush()
        _RESULT_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)
    return _RESULT_OUT


def emit(line):
    out = claim_stdout()
    out.write(json.dumps(line) + "\n")
    out.flush()


def dump_outputs(out_dir, **arrays):
    """--dump-outputs: what the timed path returned in its last step, one out_dir/<name>.npy per array, so that two builds
    can be compared output for output on the same (seeded) workload.  pose = 7 doubles, q (x, y, z, w) then t, the
    pose ilsm_register_dev leaves in place of the initial guess."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, np.float64))


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-frontend", action="store_true", help="skip the config-1-with-front-end record")
    ap.add_argument("--no-sweep", action="store_true", help="skip the config-3 (bandwidth regime) measurements")
    ap.add_argument("--no-sequence", action="store_true", help="skip config 2 (full loop on the long corridor sequence)")
    ap.add_argument("--no-sharded", action="store_true", help="skip configs 4 and 5 (sequences over the GPUs, sharded ScanContext)")
    ap.add_argument("--sequence-frames", type=int, default=2000)
    ap.add_argument("--sequence-oracle-frames", type=int, default=2000)
    ap.add_argument("--config4-frames", type=int, default=200)
    ap.add_argument("--sc-keyframes", type=int, default=100_000)
    ap.add_argument("--sc-queries", type=int, default=512)
    ap.add_argument("--sc-batch", type=int, default=64)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    run_gpu(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
