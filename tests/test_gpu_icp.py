"""K6 ICP loop verification on the GPU (ilsm_icp_align_batch): equal to the oracle byte for byte, batch == singles,
determinism across runs and cluster sizes, one launch per call, stress paths, the end-to-end loop check in the box scene,
and teardown."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
NO_CORRESPONDENCES, TRANSFORM = 5, 2
OPTS = dict(max_correspondence_distance=2.0, max_iterations=50, transformation_epsilon=1e-8, euclidean_fitness_epsilon=1e-6)


@pytest.fixture(scope="module")
def icp_oracle(oracle_mod):
    """oracle.icp: the CPU restatement of pcl::IterativeClosestPoint (oracle/ilsm_oracle_icp.cpp)."""
    from oracle import icp
    return icp


@pytest.fixture(scope="module")
def loop(ilsm):
    S = ilsm.synth
    return S.loop_keyframes(), 12


def key(r):
    return bytes(r)


def rot_angle(q1, q2):
    return 2 * np.arccos(min(1.0, abs(float(np.dot(q1, q2)))))


def test_gpu_matches_oracle(ilsm, icp_oracle, ctx, loop):
    kfs, n = loop
    S = ilsm.synth
    worst, mismatches = [0.0, 0.0, 0.0], 0
    for c in (0, 4, 9):
        tg = S.loop_submap(kfs, c, n)
        m = ctx.new_map().set_input_cloud(tg, 1.0)
        src = kfs[n + c]["src"]
        guesses = [(kfs[c]["q"], kfs[c]["t"]), (S.quat_mul(kfs[c]["q"], S.quat_from_rotvec([0, 0, 0.1])), kfs[c]["t"] + [0.5, -0.4, 0.0]),
                   ((0.0, 0.0, 0.0, 1.0), kfs[c]["t"])]
        for q0, t0 in guesses:
            for opts in (OPTS, dict(max_iterations=10), dict(OPTS, max_correspondence_distance=0.3, fitness_max_range=0.05)):
                g = ctx.icp_align(m, src, q0, t0, **opts)
                w = icp_oracle.icp_align(tg, src, q0, t0, **opts)
                assert (g.iterations, g.state, g.converged, g.n_correspondences) == (w.iterations, w.state, w.converged, w.n_correspondences)
                worst[0] = max(worst[0], float(np.abs(g.tv - w.tv).max()))
                worst[1] = max(worst[1], rot_angle(g.q, w.q))
                worst[2] = max(worst[2], abs(g.fitness - w.fitness) / max(abs(w.fitness), 1e-300))
                mismatches += bytes(g) != bytes(w)
        m.close()
    print(f"GPU vs oracle: {mismatches} results not byte-equal; max |dt| {worst[0]:.3e} m, max rotation {worst[1]:.3e} rad, "
          f"max fitness rel {worst[2]:.3e}")
    # the kernel and the oracle share every arithmetic step (DESIGN section 2): equal bytes, not a tolerance
    assert mismatches == 0


def test_batch_equals_singles_bit_for_bit(ilsm, ctx, loop):
    kfs, n = loop
    S = ilsm.synth
    maps = [ctx.new_map().set_input_cloud(S.loop_submap(kfs, c, n), 1.0) for c in (1, 5, 8)]
    empty = ctx.new_map().set_input_cloud(np.zeros((0, 3), np.float32))
    targets = [maps[0], maps[1], empty, maps[2], maps[0]]
    sources = [kfs[n + 1]["src"], kfs[n + 5]["src"][:700], kfs[n + 2]["src"], np.zeros((0, 3), np.float32), kfs[n + 8]["src"]]
    guesses = [(kfs[c]["q"], kfs[c]["t"]) for c in (1, 5, 2, 8, 1)]
    batch = ctx.icp_align_batch(targets, sources, guesses, **OPTS)
    singles = [ctx.icp_align(m, s, q, t, **OPTS) for m, s, (q, t) in zip(targets, sources, guesses)]
    assert [key(r) for r in batch] == [key(r) for r in singles]
    for r, (q, t) in ((batch[2], guesses[2]), (batch[3], guesses[3])):  # empty target, empty source
        assert (r.state, r.iterations, r.converged) == (NO_CORRESPONDENCES, 0, 0)
        assert np.array_equal(r.q, q) and np.array_equal(r.tv, t)
    assert batch[0].converged and batch[4].iterations > 0
    for m in maps + [empty]:
        m.close()


def test_deterministic_across_runs_and_cluster_sizes(ilsm, ctx, loop, tmp_path):
    kfs, n = loop
    S = ilsm.synth
    tg, src = S.loop_submap(kfs, 6, n), kfs[n + 6]["src"]
    m = ctx.new_map().set_input_cloud(tg, 1.0)
    a = ctx.icp_align(m, src, kfs[6]["q"], kfs[6]["t"], **OPTS)
    b = ctx.icp_align(m, src, kfs[6]["q"], kfs[6]["t"], **OPTS)
    assert key(a) == key(b)
    m.close()
    # a fresh process with 8-CTA clusters (the cluster size is chosen once per context from the environment)
    np.save(tmp_path / "tg.npy", tg), np.save(tmp_path / "src.npy", src)
    np.save(tmp_path / "g.npy", np.concatenate([kfs[6]["q"], kfs[6]["t"]]))
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = (f"import sys; sys.path.insert(0, {root!r}); import numpy as np, ilsm_b200 as I; c = I.Context(0); "
            f"m = c.new_map().set_input_cloud(np.load({str(tmp_path / 'tg.npy')!r}), 1.0); g = np.load({str(tmp_path / 'g.npy')!r}); "
            f"r = c.icp_align(m, np.load({str(tmp_path / 'src.npy')!r}), g[:4], g[4:], **{OPTS!r}); "
            f"open({str(tmp_path / 'r8.bin')!r}, 'wb').write(bytes(r))")
    subprocess.run([sys.executable, "-c", code], check=True, env=dict(os.environ, ILSM_SOLVE_CLUSTER="8"))
    assert (tmp_path / "r8.bin").read_bytes() == key(a)


def test_one_launch_per_call(ilsm, ctx, loop):
    kfs, n = loop
    S = ilsm.synth
    m = ctx.new_map().set_input_cloud(S.loop_submap(kfs, 2, n), 1.0)
    for opts in (dict(max_iterations=1), OPTS, dict(max_iterations=40)):
        for npairs in (1, 7):
            before = ilsm.launch_count()
            rs = ctx.icp_align_batch([m] * npairs, [kfs[n + 2]["src"]] * npairs, [(kfs[2]["q"], kfs[2]["t"])] * npairs, **opts)
            assert ilsm.launch_count() - before == 1, (opts, npairs, [r.iterations for r in rs])
    before = ilsm.launch_count()
    assert ctx.icp_align_batch([], []) == [] and ilsm.launch_count() == before
    m.close()


@pytest.mark.parametrize("gated", [False, True])
def test_stress_large_source_and_outside_box(ilsm, icp_oracle, ctx, loop, gated):
    kfs, n = loop
    S = ilsm.synth
    tg = S.loop_submap(kfs, 3, n)
    m = ctx.new_map().set_input_cloud(tg, 1.0)
    rng = np.random.default_rng(3)
    big = np.concatenate([kfs[n + 3]["src"]] * 20) + rng.normal(0, 0.02, (20 * len(kfs[n + 3]["src"]), 3)).astype(np.float32)
    assert len(big) > 100_000
    opts = dict(max_iterations=8, max_correspondence_distance=1.0 if gated else float(np.sqrt(np.finfo(np.float64).max)))
    far_t = kfs[3]["t"] + [150.0, 0.0, 0.0]  # most queries fall outside the target's box: the brute-force fallback
    for src, (q0, t0) in ((big, (kfs[3]["q"], kfs[3]["t"])), (kfs[n + 3]["src"], (kfs[3]["q"], far_t))):
        g = ctx.icp_align(m, src, q0, t0, **opts)
        w = icp_oracle.icp_align(tg, src, q0, t0, **opts)
        assert (g.iterations, g.state, g.converged, g.n_correspondences) == (w.iterations, w.state, w.converged, w.n_correspondences)
        assert bytes(g) == bytes(w), (g.tv, w.tv, g.q, w.q, g.fitness, w.fitness)
    m.close()


def test_end_to_end_loop_check(ilsm, ctx, loop):
    """ScanContext candidate -> submap -> yaw guess from the shift -> ICP -> accept on converged && fitness < threshold."""
    kfs, n = loop
    S = ilsm.synth
    threshold = 0.3
    db = ilsm.ScanContextDb(ctx)
    db.add(np.stack([db.make_scancontext(k["src"]) for k in kfs[:n]]))
    cur = kfs[n + 4]
    ids, _, dist, shifts = db.query_candidates(db.make_scancontext(cur["src"]), num_candidates=10)
    best = int(np.argmin(np.where(ids >= 0, dist, np.inf)))
    c, shift = int(ids[best]), int(shifts[best])
    assert c == 4, (ids, dist)
    m = ctx.new_map().set_input_cloud(S.loop_submap(kfs, c, n), 1.0)
    q0 = S.quat_mul(kfs[c]["q"], S.quat_from_rotvec([0.0, 0.0, np.deg2rad(6.0 * shift)]))
    r = ctx.icp_align(m, cur["src"], q0, kfs[c]["t"], **OPTS)
    dt, dr = float(np.linalg.norm(r.tv - cur["t"])), float(S.quat_angle(r.q, cur["q"]))
    print(f"revisit: shift {shift}, state {r.state}, {r.iterations} iterations, fitness {r.fitness:.4f}, error {dt:.4f} m / {np.rad2deg(dr):.3f} deg")
    assert r.converged and r.fitness < threshold and dt < 0.05 and dr < np.deg2rad(0.5)
    # two different places (opposite sides of the loop) are rejected
    far = ctx.new_map().set_input_cloud(S.loop_submap(kfs, (c + n // 2) % n, n), 1.0)
    bad = ctx.icp_align(far, cur["src"], q0, kfs[c]["t"], **OPTS)
    print(f"wrong place: state {bad.state}, fitness {bad.fitness:.4f}")
    assert not (bad.converged and bad.fitness < threshold)
    m.close(), far.close(), db.close()


def test_teardown_returns_live_bytes(ilsm, loop):
    kfs, n = loop
    before = ilsm.live_bytes()
    c = ilsm.Context(0)
    m = c.new_map().set_input_cloud(ilsm.synth.loop_submap(kfs, 0, n), 1.0)
    c.icp_align_batch([m] * 3, [kfs[n]["src"]] * 3, None, max_iterations=3)
    assert ilsm.live_bytes() != before
    m.close(), c.close()
    assert ilsm.live_bytes() == before


def test_target_of_another_context_is_rejected(ilsm, ctx, loop):
    kfs, n = loop
    other = ilsm.Context(0)
    m = other.new_map().set_input_cloud(kfs[0]["world"], 1.0)
    with pytest.raises(ilsm.IlsmError) as e:
        ctx.icp_align(m, kfs[n]["src"])
    assert e.value.code == -1 and "another context" in str(e.value)
    m.close(), other.close()
