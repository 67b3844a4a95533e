"""K6 ICP loop verification without a GPU: the oracle (oracle/ilsm_oracle_icp.cpp) against an independent numpy
restatement of pcl::IterativeClosestPoint (exact float32 1-NN, Kabsch by SVD, the state machine in Python), one
case per terminal state; non-finite points; ground-truth recovery; the ABI surface (struct layouts, argument errors)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FMAX = np.finfo(np.float64).max
NOT_CONVERGED, ITERATIONS, TRANSFORM, ABS_MSE, REL_MSE, NO_CORRESPONDENCES = range(6)


@pytest.fixture(scope="module")
def icp_oracle(oracle_mod):
    """oracle.icp: the CPU restatement of pcl::IterativeClosestPoint (oracle/ilsm_oracle_icp.cpp)."""
    from oracle import icp
    return icp


def quat_mul(a, b):
    ax, ay, az, aw = a
    bx, by, bz, bw = b
    return np.array([aw * bx + ax * bw + ay * bz - az * by, aw * by + ay * bw + az * bx - ax * bz,
                     aw * bz + az * bw + ax * by - ay * bx, aw * bw - ax * bx - ay * by - az * bz])


def quat_from_mat(R):
    from scipy.spatial.transform import Rotation
    q = Rotation.from_matrix(R).as_quat()  # x y z w
    return -q if q[3] < 0 else q


def rotate(q, v):
    """Eigen's _transformVector in float64, the operation order of the library's pose helper."""
    u = np.asarray(q[:3], np.float64)
    uv = np.cross(np.broadcast_to(u, v.shape), v)
    uv = uv + uv
    return (v + q[3] * uv) + np.cross(np.broadcast_to(u, v.shape), uv)


def transform(q, t, v):
    """pointAssociateToMap: double math, float store (a non-finite point stays non-finite)."""
    with np.errstate(invalid="ignore", over="ignore"):
        return (rotate(q, v) + t).astype(np.float32)


def flann_d2(a, b):
    """The 1-NN distance expression of FLANN's L2_Simple in float32, ((dx*dx)+(dy*dy))+(dz*dz), row by row."""
    with np.errstate(invalid="ignore", over="ignore"):
        d = [a[:, k] - b[:, k] for k in range(3)]
        return (d[0] * d[0] + d[1] * d[1]) + d[2] * d[2]


def nn1(target, moved):
    """Exact 1-NN under flann_d2, ties by (d2, index).  A fp64 k-d tree (scipy's cKDTree) gives each query its exact
    nearest distance dmin; every target point within dmin (1 + 1e-5) is a candidate (the float expression is within a
    few 1e-7 of the exact squared distance), and the candidates are ranked by (float d2, index).  A point with a
    non-finite coordinate, target or query, never takes part: j = -1 and d2 = inf where no target point does."""
    from scipy.spatial import cKDTree
    T = np.asarray(target, np.float32)[:, :3]
    live = np.flatnonzero(np.isfinite(T).all(axis=1))
    T = T[live]
    j = np.full(len(moved), -1, np.int64)
    d2 = np.full(len(moved), np.inf, np.float32)
    qs = np.flatnonzero(np.isfinite(moved).all(axis=1))
    if not len(T) or not len(qs):
        return j, d2
    tree = cKDTree(T.astype(np.float64))
    q = moved[qs].astype(np.float64)
    dmin, _ = tree.query(q, k=1)
    cand = tree.query_ball_point(q, dmin * (1 + 1e-5) + 1e-20)
    qi = np.repeat(np.arange(len(qs)), [len(c) for c in cand])
    ti = np.concatenate([np.asarray(c, np.int64) for c in cand])
    dd = flann_d2(moved[qs][qi], T[ti])
    order = np.lexsort((ti, dd, qi))
    first = order[np.r_[True, qi[order][1:] != qi[order][:-1]]]
    assert len(first) == len(qs)  # every finite query has at least its exact nearest point as a candidate
    j[qs], d2[qs] = live[ti[first]], dd[first]
    return j, d2


def np_icp(target, source, q, t, max_correspondence_distance=np.sqrt(FMAX), max_iterations=10, transformation_epsilon=0.0,
           transformation_rotation_epsilon=0.0, euclidean_fitness_epsilon=-FMAX, fitness_max_range=FMAX):
    T = np.asarray(target, np.float32)[:, :3]
    S = np.asarray(source, np.float32)[:, :3].astype(np.float64)
    q, t = np.array(q, np.float64), np.array(t, np.float64)
    rot_thr = transformation_rotation_epsilon if transformation_rotation_epsilon > 0 else 1.0 - transformation_epsilon
    gate = max_correspondence_distance * max_correspondence_distance
    prev_mse, it = FMAX, 0
    while True:
        moved = transform(q, t, S)
        j, d2 = nn1(T, moved)
        keep = (j >= 0) & (d2.astype(np.float64) <= gate)
        n = int(keep.sum())
        mse = float(np.sum(d2[keep].astype(np.float64)) / n) if n else FMAX
        if n < 3:
            state = NO_CORRESPONDENCES
            break
        p, r = moved[keep].astype(np.float64), T[j[keep]].astype(np.float64)
        mp, mr = p.mean(0), r.mean(0)
        U, _, Vt = np.linalg.svd((p - mp).T @ (r - mr))
        D = np.diag([1.0, 1.0, np.sign(np.linalg.det(Vt.T @ U.T))])
        R = Vt.T @ D @ U.T
        ti = mr - R @ mp
        q = quat_mul(quat_from_mat(R), q)
        q = q / np.linalg.norm(q)
        t = R @ t + ti
        it += 1
        if it >= max_iterations:
            state = ITERATIONS
            break
        if 0.5 * (np.trace(R) - 1.0) >= rot_thr and ti @ ti <= transformation_epsilon:
            state = TRANSFORM
            break
        if abs(mse - prev_mse) < 1e-12:
            state = ABS_MSE
            break
        if abs(mse - prev_mse) / prev_mse < euclidean_fitness_epsilon:
            state = REL_MSE
            break
        prev_mse = mse
    j, d2 = nn1(T, transform(q, t, S))
    inr = (j >= 0) & (d2.astype(np.float64) <= fitness_max_range)
    fitness = float(np.sum(d2[inr].astype(np.float64)) / inr.sum()) if inr.any() else FMAX
    return dict(q=q, t=t, iterations=it, state=state, converged=state not in (NOT_CONVERGED, NO_CORRESPONDENCES),
                n_correspondences=n, fitness=fitness, mse=mse)


def scene(seed=7, n=2000):
    """~2k points on planar patches of several orientations (every degree of freedom constrained)."""
    rng = np.random.default_rng(seed)
    pts = []
    for k in range(8):
        nrm = rng.normal(size=3)
        nrm /= np.linalg.norm(nrm)
        a = np.cross(nrm, [0.0, 0.0, 1.0] if abs(nrm[2]) < 0.9 else [1.0, 0.0, 0.0])
        a /= np.linalg.norm(a)
        b = np.cross(nrm, a)
        c = rng.uniform(-12, 12, 3)
        uv = rng.uniform(-4, 4, (n // 8, 2))
        pts.append(c + uv[:, :1] * a + uv[:, 1:] * b)
    return np.concatenate(pts).astype(np.float32)


def pair(seed=7, noise=0.01, yaw=0.08, shift=(0.35, -0.25, 0.1)):
    """target; source = the target's points under the inverse of (yaw, shift), with noise; the true pose."""
    from scipy.spatial.transform import Rotation
    T = scene(seed)
    rng = np.random.default_rng(seed + 1)
    R = Rotation.from_rotvec([0.01, -0.02, yaw]).as_matrix()
    src = ((T.astype(np.float64) - shift) @ R + rng.normal(0, noise, T.shape)).astype(np.float32)
    return T, src, quat_from_mat(R), np.asarray(shift, np.float64)


def rot_angle(q1, q2):
    d = abs(float(np.dot(q1, q2)))
    return 2 * np.arccos(min(1.0, d))


def agree(r, w):
    assert (r.iterations, r.state, bool(r.converged), r.n_correspondences) == \
        (w["iterations"], w["state"], w["converged"], w["n_correspondences"])
    assert np.abs(r.tv - w["t"]).max() <= 1e-9
    assert rot_angle(r.q, w["q"]) <= 1e-9
    assert abs(r.fitness - w["fitness"]) <= 1e-12 * abs(w["fitness"])


CASES = {
    "transform": (dict(max_iterations=60, transformation_epsilon=1e-8), TRANSFORM),
    "rel_mse": (dict(max_iterations=60, euclidean_fitness_epsilon=1e-6), REL_MSE),
    "iterations": (dict(max_iterations=3), ITERATIONS),
    "max_iterations_0": (dict(max_iterations=0), ITERATIONS),
    "gated": (dict(max_iterations=60, max_correspondence_distance=0.5, transformation_epsilon=1e-8), TRANSFORM),
    "fitness_range": (dict(max_iterations=60, transformation_epsilon=1e-8, fitness_max_range=1e-4), TRANSFORM),
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_oracle_matches_numpy_restatement(icp_oracle, case):
    opts, want_state = CASES[case]
    T, S, _, _ = pair()
    q0, t0 = np.array([0.0, 0.0, 0.0, 1.0]), np.array([0.2, -0.1, 0.0])
    r = icp_oracle.icp_align(T, S, q0, t0, **opts)
    w = np_icp(T, S, q0, t0, **opts)
    agree(r, w)
    assert r.state == want_state
    if want_state == ITERATIONS:
        assert r.converged and r.iterations == max(1, opts["max_iterations"])  # the do-while runs at least once
    if "fitness_max_range" in opts:  # the range excludes points: a smaller mean than over every point
        full = icp_oracle.icp_align(T, S, q0, t0, **{k: v for k, v in opts.items() if k != "fitness_max_range"})
        assert r.fitness < full.fitness


def test_no_correspondences_keeps_the_guess(icp_oracle):
    T, S, _, _ = pair()
    q0, t0 = np.array([0.0, 0.0, 0.0, 1.0]), np.array([3.0, 2.0, 1.0])
    r = icp_oracle.icp_align(T, S, q0, t0, max_correspondence_distance=1e-3)
    agree(r, np_icp(T, S, q0, t0, max_correspondence_distance=1e-3))
    assert r.state == NO_CORRESPONDENCES and not r.converged and r.iterations == 0
    assert np.array_equal(r.q, q0) and np.array_equal(r.tv, t0)


def test_too_few_points_and_empty_target(icp_oracle):
    T, S, _, _ = pair()
    for tgt, src in ((T, S[:2]), (T[:0], S)):
        r = icp_oracle.icp_align(tgt, src, (0, 0, 0, 1), (0.5, 0, 0))
        assert (r.state, r.iterations, r.converged) == (NO_CORRESPONDENCES, 0, 0)
        assert np.array_equal(r.tv, [0.5, 0, 0])


def test_non_finite_points_never_take_part(icp_oracle):
    """NaN / Inf target points are left out (the result equals the run without them: the finite points keep their
    order); a source point whose transform is non-finite has no correspondence, even with no gate and no range."""
    T, S, _, _ = pair()
    Tb, Sb = T.copy(), S.copy()
    bad = np.arange(3, len(T), 41)
    for k, i in enumerate(bad):
        Tb[i, k % 3] = (np.nan, np.inf, -np.inf)[k % 3]
        Sb[i + 1, (k + 1) % 3] = (np.nan, np.inf, -np.inf)[k % 3]
    Sb[7] = np.finfo(np.float32).max  # finite, but any yaw near the true one overflows its float store
    q0, t0 = np.array([0.0, 0.0, np.sin(0.03), np.cos(0.03)]), np.array([0.2, -0.1, 0.0])
    for opts in (dict(max_iterations=30, transformation_epsilon=1e-8),
                 dict(max_iterations=30, transformation_epsilon=1e-8, max_correspondence_distance=np.inf, fitness_max_range=np.inf)):
        r = icp_oracle.icp_align(Tb, Sb, q0, t0, **opts)
        agree(r, np_icp(Tb, Sb, q0, t0, **opts))
        assert bytes(r) == bytes(icp_oracle.icp_align(np.delete(Tb, bad, axis=0), Sb, q0, t0, **opts))
        assert r.converged and np.isfinite(r.fitness) and np.isfinite(r.mse)


def test_recovers_known_transform(icp_oracle):
    T, S, q_true, t_true = pair(noise=0.0)
    r = icp_oracle.icp_align(T, S, (0, 0, 0, 1), (0.2, -0.1, 0.0), max_iterations=100, transformation_epsilon=1e-14,
                             max_correspondence_distance=1.0)
    assert r.converged
    assert np.abs(r.tv - t_true).max() < 1e-6 and rot_angle(r.q, q_true) < 1e-6, (r.tv, t_true, r.q, q_true)


def test_abi_struct_sizes_match_ctypes(ilsm, tmp_path):
    from ilsm_b200 import binding as b
    src = tmp_path / "s.c"
    src.write_text('#include <stdio.h>\n#include "ilsm.h"\n'
                   'int main(void){printf("%zu %zu\\n", sizeof(ilsm_icp_opts), sizeof(ilsm_icp_result)); return 0;}\n')
    exe = tmp_path / "s"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    so, sr = map(int, subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split())
    assert (so, sr) == (C.sizeof(b.IcpOpts), C.sizeof(b.IcpResult)) == (48, 88)
    from oracle import icp
    assert (C.sizeof(icp.IcpOpts), C.sizeof(icp.IcpResult)) == (so, sr)


def test_abi_defaults_are_pcls(ilsm):
    o = ilsm.IcpOpts()
    assert o.max_correspondence_distance == np.sqrt(FMAX) and o.max_iterations == 10
    assert o.transformation_epsilon == 0 and o.transformation_rotation_epsilon == 0
    assert o.euclidean_fitness_epsilon == -FMAX and o.fitness_max_range == FMAX


def test_abi_rejects_bad_arguments_without_a_gpu(ilsm):
    """Argument errors come back as ILSM_ERR_INVALID_ARG with a message before any CUDA call (so no GPU is needed)."""
    from ilsm_b200 import binding as b
    lib = b.load_library()
    fake = C.create_string_buffer(64)  # never dereferenced on these paths
    ctx, vp = C.cast(fake, C.c_void_p), C.c_void_p
    maps = (vp * 2)(ctx.value, ctx.value)
    pts = np.zeros((8, 3), np.float32)
    res = (b.IcpResult * 2)()
    good = np.array([0, 4, 8], np.int32)
    o = b.IcpOpts()
    call = lambda c, m, n, offs, opts=o: lib.ilsm_icp_align_batch(c, m, n, pts.ctypes.data, offs.ctypes.data, 12, None,
                                                                  C.byref(opts), res)
    assert call(None, maps, 2, good) == -1
    assert b"null ctx" in lib.ilsm_last_error()
    assert call(ctx, maps, -1, good) == -1
    assert call(ctx, None, 2, good) == -1
    assert call(ctx, maps, 2, np.array([4, 0, 8], np.int32)) == -1
    assert b"offsets decrease" in lib.ilsm_last_error()
    assert call(ctx, maps, 2, good, b.IcpOpts(max_iterations=-1)) == -1
    assert b"max_iterations" in lib.ilsm_last_error()
    assert lib.ilsm_icp_align_batch(ctx, maps, 2, None, good.ctypes.data, 12, None, None, res) == -1
    assert b"null source" in lib.ilsm_last_error()
    assert call(ctx, maps, 0, good) == 0  # an empty batch: nothing to launch
