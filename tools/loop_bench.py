"""Loop closure per keyframe: one ilsm_loop_add_keyframe call against a resident keyframe store, and the same steps
composed from the existing entry points on the host (the hand-written loopClosureThread body of INTEGRATION section 7a).

Workload: the 24 keyframes of synth.loop_keyframes() replicated with N(0, 2 cm) jitter into databases of 1 k and 10 k
keyframes (default options: exclude_recent 50, tree period 50, 10 candidates, threshold 0.13).  Then, one call at a time
with a host clock around each (every call ends in a synchronisation): 20 calls with no loop (frames of another scene,
ScanContext distance > 0.4 to everything stored) and 20 verified calls (jittered revisits of stored places).  The
composition runs on the same inputs: make_scancontext + add + voxelgrid + query_candidates, and for a loop the numpy
world transform of the submap, voxelgrid, a map build and icp_align.  Median and p90 per kind, the card's name and power
limit read in the same run.  Writes loop_bench.json under --out (default profiles/)."""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


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


def stats(ts):
    import numpy as np
    a = np.asarray(ts) * 1e3
    return {"calls": len(a), "median_ms": round(float(np.median(a)), 4), "p90_ms": round(float(np.percentile(a, 90)), 4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1000,10000")
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    a = ap.parse_args()
    import numpy as np
    import ilsm_b200 as ilsm
    from test_gpu_loop import Composition
    S = ilsm.synth
    kfs = S.loop_keyframes()
    other = S.Scene(seed=S.SEED_MAP + 991)
    far = []
    for i in range(4):  # another scene: no stored place is near
        q = S.quat_from_rotvec([0.0, 0.0, 0.7 * i])
        cloud, _ = S.make_frame(other, q, np.array([5.0 * i - 7.0, 3.0, 1.5]), seed=0x5EED2000 + i)
        far.append((S.voxel_centroid_np(cloud[np.any(cloud[:, :3] != 0, axis=1), :3], 0.4), q, np.array([5.0 * i - 7.0, 3.0, 1.5])))
    rng = np.random.default_rng(11)

    def jittered(kf):
        return kf["src"] + rng.normal(0, 0.02, kf["src"].shape).astype(np.float32), kf["q"], kf["t"]

    ctx = ilsm.Context(0)
    out = {"workload": "synth.loop_keyframes x jitter; default ilsm_loop_opts", **device_info(), "runs": []}
    for size in [int(s) for s in a.sizes.split(",")]:
        loop, comp = ilsm.LoopClosure(ctx), Composition(ilsm, ctx)
        t0 = time.perf_counter()
        for i in range(size):
            cl, q, t = jittered(kfs[i % len(kfs)])
            loop.add_keyframe(cl, q, t)
            comp.fill(cl, q, t)
        fill_s = time.perf_counter() - t0
        rec = {"keyframes": size, "fill_s": round(fill_s, 1)}
        for kind, inputs in (("no_loop", [far[i % len(far)] for i in range(a.calls)]),
                             ("verified", [jittered(kfs[i % len(kfs)]) for i in range(a.calls)])):
            th, tc, verified = [], [], 0
            for cl, q, t in inputs:
                t0 = time.perf_counter()
                r = loop.add_keyframe(cl, q, t)
                th.append(time.perf_counter() - t0)
                t0 = time.perf_counter()
                w = comp.add(cl, q, t)
                tc.append(time.perf_counter() - t0)
                verified += r.verified
                assert r.verified == w["verified"] and r.loop_id == w["loop_id"], (kind, r.loop_id, w["loop_id"])
            rec[kind] = {"handle": stats(th), "composition": stats(tc), "verified_calls": verified}
        out["runs"].append(rec)
        print(json.dumps(rec), flush=True)
        loop.close(), comp.close()
    ctx.close()
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "loop_bench.json"), "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps({k: out[k] for k in ("device", "nvidia_smi")}))


if __name__ == "__main__":
    main()
