"""K7 loop closure per keyframe (ilsm_loop) on the GPU: equal byte for byte to the same steps run through the existing
entry points (ScanContextDb.query_candidates under SCManager's state machine restated in Python, a numpy world transform,
ctx.voxelgrid, a map build, ctx.icp_align), revisits found and accepted, the yaw convention, a wrong place rejected, tree
staleness, launch counts, host == device input, determinism, pool growth and teardown."""
import math
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
N = 12  # keyframes per lap of synth.loop_keyframes()
ICP = dict(max_correspondence_distance=2.0, max_iterations=50, transformation_epsilon=1e-8, euclidean_fitness_epsilon=1e-6)


@pytest.fixture(scope="module")
def kfs(ilsm):
    return ilsm.synth.loop_keyframes()


def xyzi(cloud):
    a = np.asarray(cloud, np.float32)
    return np.concatenate([a[:, :3], np.zeros((len(a), 1), np.float32)], axis=1)


def rotate(q, v):
    """Eigen's _transformVector in float64, quat_rotate's operation order."""
    u = np.asarray(q[:3], np.float64)
    uv = np.cross(np.broadcast_to(u, v.shape), v)
    uv = uv + uv
    return (v + q[3] * uv) + np.cross(np.broadcast_to(u, v.shape), uv)


class Composition:
    """The handle's steps through the existing entry points, the state machine of Scancontext.cpp:253-344 in Python."""

    def __init__(self, ilsm, ctx, exclude_recent=50, tree_period=50, sc_dist_threshold=0.13, num_candidates=10, submap_half=2,
                 leaf=0.4, cell=1.0, fitness_threshold=0.3):
        self.S, self.ctx, self.db = ilsm.synth, ctx, ilsm.ScanContextDb(ctx)
        self.er, self.tp, self.thr, self.k, self.h = exclude_recent, tree_period, sc_dist_threshold, num_candidates, submap_half
        self.leaf, self.cell, self.fit = leaf, cell, fitness_threshold
        self.store, self.counter, self.n_search = [], 0, 0
        self.lc = ilsm.launch_count

    def fill(self, cloud, q, t):
        """Store a keyframe and advance the state machine; returns (its descriptor, whether a search is due)."""
        a = xyzi(cloud)
        desc = self.db.make_scancontext(a)
        self.db.add(desc)
        self.store.append((self.ctx.voxelgrid(a, self.leaf), np.asarray(q, np.float64), np.asarray(t, np.float64)))
        size = len(self.db)
        if size < self.er + 1:
            return desc, False
        if self.counter % self.tp == 0:
            self.n_search = size - self.er
        self.counter += 1
        return desc, True

    def add(self, cloud, q, t):
        desc, search = self.fill(cloud, q, t)
        size = len(self.db)
        out = dict(loop_id=-1, nn_id=-1, shift=0, sc_dist=0.0, verified=0, submap_points=0, icp=None)
        if not search:
            return out
        ids, _, dist, sh = self.db.query_candidates(desc, self.k, self.n_search)
        best, arg, align = 10000000.0, 0, 0
        for ci, cd, cs in zip(ids, dist, sh):
            if ci >= 0 and cd < best:
                best, arg, align = float(cd), int(ci), int(cs)
        out.update(nn_id=arg, shift=align, sc_dist=best)
        if not best < self.thr:
            return out
        lo, hi = max(0, arg - self.h), min(arg + self.h, size - self.er - 1)
        parts = []
        for j in range(lo, hi + 1):
            p, qj, tj = self.store[j]
            w = p.copy()
            with np.errstate(invalid="ignore", over="ignore"):
                w[:, :3] = (rotate(qj, p[:, :3].astype(np.float64)) + tj).astype(np.float32)
            parts.append(w)
        world = np.concatenate(parts)
        b0 = self.lc()
        sub = self.ctx.voxelgrid(world, self.leaf) if len(world) else np.zeros((0, 4), np.float32)
        self.submap_vg_launches = self.lc() - b0
        m = self.ctx.new_map()
        b0 = self.lc()
        m.set_input_cloud(sub, self.cell)
        self.build_launches = self.lc() - b0
        yaw = float(np.float32(align * 6.0 * math.pi / 180.0))
        qc, tc = self.store[arg][1], self.store[arg][2]
        g = self.S.quat_mul(qc, [0.0, 0.0, math.sin(-yaw * 0.5), math.cos(-yaw * 0.5)])
        r = self.ctx.icp_align(m, self.store[-1][0], g, tc, **ICP)
        m.close()
        out.update(loop_id=arg, verified=1, submap_points=len(sub), submap_first=lo, submap_last=hi, icp=bytes(r),
                   accepted=int(bool(r.converged) and r.fitness < self.fit))
        return out

    def close(self):
        self.db.close()


def agree(g, w):
    assert (g.loop_id, g.nn_id, g.shift, g.sc_dist, g.verified, g.submap_points) == \
        (w["loop_id"], w["nn_id"], w["shift"], w["sc_dist"], w["verified"], w["submap_points"]), (g.keyframe_id, w)
    if w["verified"]:
        assert (g.submap_first, g.submap_last, g.accepted) == (w["submap_first"], w["submap_last"], w["accepted"])
        assert bytes(g.icp) == w["icp"], g.keyframe_id


def run_both(ilsm, ctx, kfs, **opts):
    loop, comp = ilsm.LoopClosure(ctx, **opts), Composition(ilsm, ctx, **opts)
    got = []
    for i, kf in enumerate(kfs):
        g, w = loop.add_keyframe(kf["src"], kf["q"], kf["t"]), comp.add(kf["src"], kf["q"], kf["t"])
        assert g.keyframe_id == i and len(loop) == i + 1
        agree(g, w)
        got.append(g)
    loop.close(), comp.close()
    return got


@pytest.mark.parametrize("tree_period", [1, 4])
@pytest.mark.parametrize("threshold", [0.13, 0.3])
def test_equals_the_composition_byte_for_byte(ilsm, ctx, kfs, tree_period, threshold):
    got = run_both(ilsm, ctx, kfs, exclude_recent=6, tree_period=tree_period, sc_dist_threshold=threshold)
    assert [g.nn_id for g in got[:6]] == [-1] * 6  # early returns
    assert any(g.verified for g in got)


def rel_truth(S, kfs, c, k):
    qc, tc, qk, tk = kfs[c]["q"], kfs[c]["t"], kfs[k]["q"], kfs[k]["t"]
    qi = S.quat_inv(qc)
    return S.quat_mul(qi, qk), S.quat_to_mat(qi) @ (tk - tc)


def assert_close_to_truth(S, r, kf, q_rel, t_rel):
    assert r.accepted and r.icp.converged
    assert np.linalg.norm(r.icp.tv - kf["t"]) < 0.05 and S.quat_angle(r.icp.q, kf["q"]) < np.deg2rad(0.5)
    assert np.linalg.norm(r.tv - t_rel) < 0.05 and S.quat_angle(r.q, q_rel) < np.deg2rad(0.5)


def test_revisits_are_found_and_accepted(ilsm, ctx, kfs):
    S = ilsm.synth
    loop = ilsm.LoopClosure(ctx, exclude_recent=6, tree_period=1, sc_dist_threshold=0.3)
    res = [loop.add_keyframe(kf["src"], kf["q"], kf["t"]) for kf in kfs]
    assert all(r.loop_id == -1 for r in res[:N])
    for k in range(N):
        r = res[N + k]
        assert r.loop_id == k and r.verified, (k, r.loop_id, r.sc_dist)
        assert 0.09 < r.sc_dist < 0.19
        assert_close_to_truth(S, r, kfs[N + k], *rel_truth(S, kfs, k, N + k))
        print(f"lap-2 keyframe {k}: dist {r.sc_dist:.4f} shift {r.shift} fitness {r.icp.fitness:.4f} "
              f"error {np.linalg.norm(r.icp.tv - kfs[N + k]['t']):.4f} m")
    loop.close()


def test_default_threshold(ilsm, ctx, kfs):
    loop = ilsm.LoopClosure(ctx, exclude_recent=6, tree_period=1)
    assert ilsm.LoopOpts().sc_dist_threshold == 0.13
    res = [loop.add_keyframe(kf["src"], kf["q"], kf["t"]) for kf in kfs]
    assert [i for i, r in enumerate(res) if r.loop_id >= 0] == [N + 6]
    assert res[N + 6].loop_id == 6 and res[N + 6].accepted
    assert res[N + 7].nn_id == 7 and res[N + 5].nn_id == 5 and res[N + 7].sc_dist > 0.13 and res[N + 5].sc_dist > 0.13
    loop.close()


@pytest.mark.parametrize("yaw_deg", [30.0, -30.0, 90.0])
def test_yaw_convention(ilsm, ctx, kfs, yaw_deg):
    S = ilsm.synth
    loop = ilsm.LoopClosure(ctx, exclude_recent=6, tree_period=1, sc_dist_threshold=0.3)
    for kf in kfs[:N]:
        loop.add_keyframe(kf["src"], kf["q"], kf["t"])
    # 0.1 m nearer the loop centre: from 0.1 m further out, the ICP of the -30 degree revisit stops (TRANSFORM after 7
    # iterations) 8 cm from the truth -- the settings' early stop, the same on the CPU oracle; the guess is right either way
    rv = S.revisit_keyframe(kfs[4], yaw_deg)
    r = loop.add_keyframe(rv["src"], rv["q"], rv["t"])
    assert r.loop_id == 4 and r.shift == {30.0: 55, -30.0: 5, 90.0: 45}[yaw_deg]
    qi = S.quat_inv(kfs[4]["q"])
    assert_close_to_truth(S, r, rv, S.quat_mul(qi, rv["q"]), S.quat_to_mat(qi) @ (rv["t"] - kfs[4]["t"]))
    loop.close()


def test_wrong_place_is_verified_and_rejected(ilsm, ctx, kfs):
    loop = ilsm.LoopClosure(ctx, exclude_recent=6, tree_period=1, sc_dist_threshold=1.0)
    res = [loop.add_keyframe(kf["src"], kf["q"], kf["t"]) for kf in kfs[:N]]
    r = res[11]
    assert (r.loop_id, r.shift, r.verified, r.accepted) == (5, 55, 1, 0)
    assert abs(r.sc_dist - 0.5954) < 1e-3 and r.icp.converged and r.icp.fitness > 1.0
    assert np.array_equal(r.q, np.zeros(4)) and np.array_equal(r.tv, np.zeros(3))  # filled only when accepted
    loop.close()


def test_stale_tree_equals_the_restatement(ilsm, ctx, kfs):
    """A tree refreshed every 8th search misses counterparts the newest keyframes would offer; the handle misses them too."""
    got = run_both(ilsm, ctx, kfs, exclude_recent=6, tree_period=8, sc_dist_threshold=0.3)
    assert got[N + 1].loop_id != 1  # the tree of keyframe 13 holds keyframe 0 only
    assert got[N + 6].loop_id == 6


def test_launch_counts(ilsm, ctx, kfs):
    """No loop: exactly the launches of descriptor + append + VoxelGrid + candidates through the existing entry points (no
    gather, no ICP); a verified keyframe adds one gather, the submap VoxelGrid, one map build and exactly one ICP kernel."""
    loop = ilsm.LoopClosure(ctx, exclude_recent=6, tree_period=1, sc_dist_threshold=0.3)
    comp = Composition(ilsm, ctx, exclude_recent=6, tree_period=1, sc_dist_threshold=0.3)
    lc = ilsm.launch_count
    verified = 0
    for i, kf in enumerate(kfs):
        b0 = lc()
        r = loop.add_keyframe(kf["src"], kf["q"], kf["t"])
        handle = lc() - b0
        b0 = lc()
        comp.add(kf["src"], kf["q"], kf["t"])
        composed = lc() - b0
        if not r.verified:
            assert handle == composed, i
            continue
        verified += 1
        vg = comp.submap_vg_launches
        store_detect = composed - vg - comp.build_launches - 1  # the composition's ICP: one launch
        build = handle - store_detect - 1 - vg - 1              # gather and ICP: one launch each
        assert build in (3, 4), (i, handle, composed, vg)       # count, alloc, scatter (+ a table clear)
    assert verified == N
    loop.close(), comp.close()


def feed(loop, kfs, dev=False, stride_floats=4):
    import torch
    out = []
    for kf in kfs:
        a = np.zeros((len(kf["src"]), stride_floats), np.float32)
        a[:, :3] = kf["src"]
        if dev:
            t = torch.from_numpy(a).cuda()
            torch.cuda.synchronize()
            out.append(bytes(loop.add_keyframe_dev(t, kf["q"], kf["t"])))
        else:
            out.append(bytes(loop.add_keyframe(a, kf["q"], kf["t"])))
    return out


@pytest.mark.parametrize("stride_floats", [4, 8])
def test_host_form_equals_device_form(ilsm, ctx, kfs, stride_floats):
    runs = []
    for dev in (False, True):
        loop = ilsm.LoopClosure(ctx, exclude_recent=6, tree_period=1, sc_dist_threshold=0.3)
        runs.append(feed(loop, kfs, dev, stride_floats))
        loop.close()
    assert runs[0] == runs[1]
    assert sum(ilsm.LoopResult.from_buffer_copy(b).accepted for b in runs[0]) == N


def test_deterministic_across_runs_and_cluster_sizes(ilsm, ctx, kfs, tmp_path):
    def once(c):
        loop = ilsm.LoopClosure(c, exclude_recent=6, tree_period=1, sc_dist_threshold=0.3)
        r = feed(loop, kfs)
        loop.close()
        return r
    a, b = once(ctx), once(ctx)
    assert a == b
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = (f"import sys; sys.path.insert(0, {root!r}); sys.path.insert(0, {os.path.dirname(os.path.abspath(__file__))!r}); "
            f"import ilsm_b200 as I, test_gpu_loop as T; c = I.Context(0); l = I.LoopClosure(c, exclude_recent=6, tree_period=1, "
            f"sc_dist_threshold=0.3); r = T.feed(l, I.synth.loop_keyframes()); open({str(tmp_path / 'r8.bin')!r}, 'wb').write(b''.join(r))")
    subprocess.run([sys.executable, "-c", code], check=True, env=dict(os.environ, ILSM_SOLVE_CLUSTER="8"))
    assert (tmp_path / "r8.bin").read_bytes() == b"".join(a)


def test_pool_growth_and_teardown(ilsm, kfs):
    S = ilsm.synth
    before = ilsm.live_bytes()
    c = ilsm.Context(0)
    loop, comp = ilsm.LoopClosure(c, tree_period=1), Composition(ilsm, c, tree_period=1)
    rng = np.random.default_rng(5)
    seq = []
    for i in range(300):  # the 24 keyframes replicated with jitter: the pool and the descriptor table grow several times
        kf = kfs[i % len(kfs)]
        seq.append((kf["src"] + rng.normal(0, 0.02, kf["src"].shape).astype(np.float32), kf["q"], kf["t"]))
    rv = S.revisit_keyframe(kfs[0], 30.0)
    seq.append((rv["src"], rv["q"], rv["t"]))
    for i, (cl, q, t) in enumerate(seq):
        g = loop.add_keyframe(cl, q, t)
        w = comp.add(cl, q, t)
        if i == len(seq) - 1:
            agree(g, w)
            assert g.verified and g.accepted
    assert len(loop) == 301
    comp.close(), loop.close(), c.close()
    assert ilsm.live_bytes() == before
