"""K6 ICP loop verification at its edges on the GPU.  Every case runs three implementations on the same inputs: the
kernel (icp_cluster_kernel), the oracle (oracle/ilsm_oracle_icp.cpp) and the independent numpy restatement
(test_icp_cpu.np_icp: exact float 1-NN, Kabsch by SVD).  The kernel and the oracle share every arithmetic step (operation
order, float store, reduction tree, Horn solve), so their results must be equal byte for byte; against the numpy
restatement, states, iteration and correspondence counts are equal, the pose agrees to 1e-9 m / 1e-9 rad and the
fitness to 1e-12 relative.  Cases: tile and cluster shapes, every terminal state, correspondence gates at and next to
float-representable d2, option edges (zero, negative, NaN), (d2, index) ties, cell sizes, rotations near 180 degrees,
kilometre-scale coordinates, rank-deficient fits, non-finite points, the device-pointer entry point, source strides,
large mixed batches and rebuilt target handles."""
import ctypes as C
import time

import numpy as np
import pytest

from test_icp_cpu import (ABS_MSE, FMAX, ITERATIONS, NO_CORRESPONDENCES, REL_MSE, TRANSFORM, nn1, np_icp, quat_mul,
                          transform)

pytestmark = pytest.mark.gpu

OPTS = dict(max_correspondence_distance=1.0, max_iterations=40, transformation_epsilon=1e-10, euclidean_fitness_epsilon=1e-7)
IDENTITY = ((0.0, 0.0, 0.0, 1.0), (0.0, 0.0, 0.0))
WORST = dict(dt=0.0, drot=0.0, dfit=0.0, dpts=0.0, ref_s=0.0, cases=0)


@pytest.fixture(scope="module")
def icp_oracle(oracle_mod):
    from oracle import icp
    return icp


@pytest.fixture(scope="module", autouse=True)
def report(request):
    """The worst GPU-vs-reference deviations of the module and the time the numpy reference took."""
    yield
    line = (f"ICP edges, GPU vs numpy reference over {WORST['cases']} runs: max |dt| {WORST['dt']:.3e} m, max rotation "
            f"{WORST['drot']:.3e} rad, max fitness rel {WORST['dfit']:.3e}, max point |d| {WORST['dpts']:.3e} m; "
            f"reference time {WORST['ref_s']:.1f} s")
    tr = request.config.pluginmanager.get_plugin("terminalreporter")
    tr.write_line(line) if tr is not None else print(line)


# ---------------------------------------------------------------------------------------------------------------------
# scenes
# ---------------------------------------------------------------------------------------------------------------------
def quat_z(deg):
    h = np.deg2rad(deg) / 2
    return np.array([0.0, 0.0, np.sin(h), np.cos(h)])


def planes(seed, n, k=8):
    """n points on k square patches (8 m) of random orientation within 12 m of the origin: every degree of freedom is
    constrained.  The patches depend on the seed only, the samples on (seed, n)."""
    rng = np.random.default_rng(seed)
    frames = []
    for _ in range(k):
        nrm = rng.normal(size=3)
        nrm /= np.linalg.norm(nrm)
        a = np.cross(nrm, [0.0, 0.0, 1.0] if abs(nrm[2]) < 0.9 else [1.0, 0.0, 0.0])
        a /= np.linalg.norm(a)
        frames.append((rng.uniform(-12, 12, 3), a, np.cross(nrm, a)))
    rng = np.random.default_rng([seed, n])
    uv = rng.uniform(-4, 4, (n, 2))
    c, a, b = (np.array([f[i] for f in frames])[np.arange(n) % k] for i in range(3))
    return (c + uv[:, :1] * a + uv[:, 1:] * b).astype(np.float32)


def make_pair(n_src, n_tgt=1200, seed=11, noise=0.005, q_true=None, shift=(0.3, -0.2, 0.05), rng_seed=0):
    """target: n_tgt points on the patches; source: n_src other samples of the same patches seen from the pose
    (q_true, shift), with noise.  Returns (target, source, q_true, shift)."""
    from scipy.spatial.transform import Rotation
    q_true = np.asarray(q_true if q_true is not None else Rotation.from_rotvec([0.01, -0.02, 0.05]).as_quat(), np.float64)
    R = Rotation.from_quat(q_true).as_matrix()
    T = planes(seed, n_tgt)
    P = planes(seed, n_src + 7)[:n_src].astype(np.float64)  # another sample of the same patches
    rng = np.random.default_rng(rng_seed)
    S = ((P - shift) @ R + rng.normal(0, noise, P.shape)).astype(np.float32)
    return T, S, q_true, np.asarray(shift, np.float64)


def lattice(n, spacing, seed=None):
    g = np.stack(np.meshgrid(*[np.arange(n)] * 3, indexing="ij"), -1).reshape(-1, 3).astype(np.float32) * np.float32(spacing)
    return g[np.random.default_rng(seed).permutation(len(g))] if seed is not None else g


def flann_d2(a, b):
    d = (np.asarray(a, np.float32) - np.asarray(b, np.float32)).astype(np.float32)
    return (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]


def point_at_d2(p, want):
    """A float point q with the 1-NN distance expression d2(q, p) == want exactly (want: a float32): x moves by about
    sqrt(want), y by up to a few thousand ulps for the last bits.  p[0] == 0 and p[1] > 0."""
    p = np.asarray(p, np.float32)
    want = np.float32(want)
    bx = np.float32(np.sqrt(want)).view(np.int32) + np.arange(-64, 65, dtype=np.int32)
    by = p[1].view(np.int32) + np.arange(0, 4096, dtype=np.int32)
    xs, ys = bx.view(np.float32), by.view(np.float32)
    dx, dy = xs - p[0], ys - p[1]
    d2 = (dx[:, None] * dx[:, None] + dy[None, :] * dy[None, :]) + np.float32(0) * np.float32(0)
    i, j = np.argwhere(d2 == want)[0]
    q = np.array([xs[i], ys[j], p[2]], np.float32)
    assert flann_d2(q, p) == want
    return q


# ---------------------------------------------------------------------------------------------------------------------
# the three-way check
# ---------------------------------------------------------------------------------------------------------------------
def rot_dist(q1, q2):
    """Angle of the rotation between two unit quaternions, accurate for small angles."""
    q1, q2 = np.asarray(q1, np.float64), np.asarray(q2, np.float64)
    s = 1.0 if np.dot(q1, q2) >= 0 else -1.0
    return 4.0 * np.arcsin(min(1.0, np.linalg.norm(q1 - s * q2) / 2.0))


def fields(r):
    return (tuple(r.q_xyzw), tuple(r.t), r.fitness, r.mse, r.iterations, r.state, r.converged, r.n_correspondences)


def same_bytes(g, w):
    assert bytes(g) == bytes(w), f"GPU != oracle:\n  GPU    {fields(g)}\n  oracle {fields(w)}"


def agree_ref(g, r, src=None):
    """GPU result g vs numpy reference dict r.  src given: the pose is unobservable about a line, so compare the
    transformed source points (fp64) instead of the pose."""
    assert (g.iterations, g.state, bool(g.converged), g.n_correspondences) == \
        (r["iterations"], r["state"], r["converged"], r["n_correspondences"]), (fields(g), r)
    if src is not None:
        S = np.asarray(src, np.float32)[:, :3].astype(np.float64)
        from test_icp_cpu import rotate
        dp = float(np.abs((rotate(g.q, S) + g.tv) - (rotate(r["q"], S) + r["t"])).max()) if len(S) else 0.0
        WORST["dpts"] = max(WORST["dpts"], dp)
        assert dp <= 1e-9
        mse_ok = g.mse == r["mse"] or abs(g.mse - r["mse"]) <= 1e-12 * abs(r["mse"])
        assert mse_ok, (g.mse, r["mse"])
    else:
        dt, dr = float(np.abs(g.tv - r["t"]).max()), rot_dist(g.q, r["q"])
        WORST["dt"], WORST["drot"] = max(WORST["dt"], dt), max(WORST["drot"], dr)
        assert dt <= 1e-9 and dr <= 1e-9, (dt, dr)
    if r["fitness"] == FMAX:
        assert g.fitness == FMAX
    else:
        df = abs(g.fitness - r["fitness"]) / abs(r["fitness"]) if r["fitness"] else abs(g.fitness)
        WORST["dfit"] = max(WORST["dfit"], df)
        assert df <= 1e-12, (g.fitness, r["fitness"])


def reference(tgt, src, q0, t0, **opts):
    t = time.perf_counter()
    r = np_icp(tgt, src, q0, t0, **opts)
    WORST["ref_s"] += time.perf_counter() - t
    WORST["cases"] += 1
    return r


def gpu(ctx, tgt, src, q0, t0, cell=1.0, **opts):
    m = ctx.new_map().set_input_cloud(tgt, cell)
    try:
        return ctx.icp_align(m, src, q0, t0, **opts)
    finally:
        m.close()


def check(ctx, icp_oracle, tgt, src, q0=IDENTITY[0], t0=IDENTITY[1], cell=1.0, points=False, **opts):
    """GPU == oracle byte for byte, GPU ~ numpy reference; returns (GPU result, reference dict)."""
    g = gpu(ctx, tgt, src, q0, t0, cell, **opts)
    same_bytes(g, icp_oracle.icp_align(tgt, src, q0, t0, **opts))
    r = reference(tgt, src, q0, t0, **opts)
    agree_ref(g, r, src if points else None)
    return g, r


def guess_of(q_true, t_true):
    """A guess about 3 degrees and 0.3 m off the true pose."""
    from scipy.spatial.transform import Rotation
    return quat_mul(Rotation.from_rotvec([0.0, 0.01, 0.05]).as_quat(), q_true), t_true + [0.2, -0.25, 0.1]


# ---------------------------------------------------------------------------------------------------------------------
# tile and cluster shapes
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_src", [1, 2, 3, 4, 31, 32, 33, 255, 256, 257, 7 * 256, 8 * 256, 8 * 256 + 1, 16 * 256,
                                   16 * 256 + 1, 40 * 256 + 17])
def test_tile_and_cluster_shapes(ctx, icp_oracle, n_src):
    """One tile or many: fewer tiles than CTAs, exactly 8 or 16 tiles (one per CTA of either cluster size), a ragged
    last tile, and 1-3 points."""
    T, S, q, t = make_pair(n_src)
    q0, t0 = guess_of(q, t)
    g, _ = check(ctx, icp_oracle, T, S, q0, t0, **OPTS)
    if n_src < 3:
        assert (g.state, g.iterations, g.converged) == (NO_CORRESPONDENCES, 0, 0)
        assert np.array_equal(g.q, q0) and np.array_equal(g.tv, t0)
    else:
        assert g.iterations >= 1 and g.state in (TRANSFORM, REL_MSE, ABS_MSE, ITERATIONS)


# ---------------------------------------------------------------------------------------------------------------------
# terminal states
# ---------------------------------------------------------------------------------------------------------------------
STATES = {
    "transform": (dict(max_iterations=60, transformation_epsilon=1e-8), TRANSFORM),
    "transform_rotation_eps": (dict(max_iterations=60, transformation_epsilon=1e-6, transformation_rotation_epsilon=1 - 1e-9),
                               TRANSFORM),
    "rel_mse": (dict(max_iterations=60, euclidean_fitness_epsilon=1e-3), REL_MSE),
    "iterations_0": (dict(max_iterations=0), ITERATIONS),
    "iterations_1": (dict(max_iterations=1), ITERATIONS),
    "iterations_3": (dict(max_iterations=3), ITERATIONS),
    "no_corr_at_entry": (dict(max_correspondence_distance=0.05), NO_CORRESPONDENCES),
}


@pytest.mark.parametrize("case", list(STATES))
def test_terminal_states(ctx, icp_oracle, case):
    opts, want = STATES[case]
    T, S, q, t = make_pair(3000, n_tgt=2000)
    q0, t0 = guess_of(q, t)
    if case == "no_corr_at_entry":
        t0 = t0 + [3.0, 0.0, 0.0]
    g, _ = check(ctx, icp_oracle, T, S, q0, t0, **opts)
    assert g.state == want
    if want == ITERATIONS:
        assert g.iterations == max(1, opts["max_iterations"]) and g.converged  # a do-while: 0 still runs once
    if case == "no_corr_at_entry":
        assert g.iterations == 0 and np.array_equal(g.q, q0) and np.array_equal(g.tv, t0)
    if case == "transform_rotation_eps":  # a stricter rotation threshold than 1 - transformation_epsilon ends it later
        g2 = gpu(ctx, T, S, q0, t0, **dict(opts, transformation_rotation_epsilon=0.0))
        assert g2.state == TRANSFORM and g2.iterations < g.iterations


def test_abs_mse_on_an_exact_rigid_copy(ctx, icp_oracle):
    """A noise-free source that is the target moved by a float-exact translation: the MSE stops changing."""
    T = planes(5, 1500)
    S = (T - np.float32([0.125, -0.25, 0.0625])).astype(np.float32)
    g, _ = check(ctx, icp_oracle, T, S, max_correspondence_distance=1.0, max_iterations=50)
    assert g.state == ABS_MSE and g.iterations >= 2
    assert g.mse < 1e-12


# Few-point source whose first fit carries it out of the gate.  The seed was found with the numpy reference; its three
# first correspondences have three different target points, so the fit is determined (a seed with two on one target
# point leaves the rotation about that pair's line free).
NO_CORR_LATE_SEED = 7078


def few_point_escape(seed):
    rng = np.random.default_rng(seed)
    T = rng.uniform(-1, 1, (6, 3)).astype(np.float32)
    S = (T[:4] + rng.normal(0, 0.3, (4, 3))).astype(np.float32)
    return T, S, dict(max_correspondence_distance=0.35, max_iterations=20)


def test_no_correspondences_after_an_iteration(ctx, icp_oracle):
    T, S, opts = few_point_escape(NO_CORR_LATE_SEED)
    g, _ = check(ctx, icp_oracle, T, S, **opts)
    assert g.state == NO_CORRESPONDENCES and g.iterations >= 1 and not g.converged


# ---------------------------------------------------------------------------------------------------------------------
# gates
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cell", [0.25, 1.0])
def test_gate_at_a_representable_d2(ctx, icp_oracle, cell):
    """max_correspondence_distance 0.5: offsets of exactly 0.5 give d2 == 0.25 == the gate, and are kept (<=); offsets
    one float above are not."""
    T = lattice(5, 2.0, seed=1)
    S = T.copy()
    axis = np.arange(len(T)) % 3
    S[np.arange(len(T)), axis] += np.float32(0.5)
    out = np.arange(len(T)) % 4 == 3
    S[out, axis[out]] = np.nextafter(S[out, axis[out]], np.float32(np.inf))
    assert (flann_d2(S[~out], T[~out]) == 0.25).all() and (flann_d2(S[out], T[out]) > 0.25).all()
    g, _ = check(ctx, icp_oracle, T, S, cell=cell, max_correspondence_distance=0.5, max_iterations=1)
    assert g.n_correspondences == int((~out).sum())


@pytest.mark.parametrize("cell", [0.05, 1.0])
@pytest.mark.parametrize("dist", [0.1, 0.3])
def test_gate_whose_square_is_not_a_float(ctx, icp_oracle, dist, cell):
    """dist^2 is not a float: the largest float d2 <= dist^2 is kept and the next one is not, whichever way the float
    rounding of dist^2 goes (0.1^2 rounds down, 0.3^2 up), so the k-NN cut-off (rounded up) must not lose the kept ones."""
    gate = dist * dist
    below = np.float32(gate) if float(np.float32(gate)) <= gate else np.nextafter(np.float32(gate), np.float32(0))
    above = np.nextafter(below, np.float32(1))
    assert float(below) <= gate < float(above)
    T = np.zeros((16, 3), np.float32)  # x = 0, y and z on a 3 m grid: no other target point near any source point
    T[:, 1:] = np.stack(np.meshgrid(np.arange(4), np.arange(4), indexing="ij"), -1).reshape(-1, 2) * 3.0 + 2.0
    wants = [below if k % 2 == 0 else above for k in range(16)]
    S = np.stack([point_at_d2(p, w) for p, w in zip(T, wants)])
    g, _ = check(ctx, icp_oracle, T, S, cell=cell, max_correspondence_distance=dist, max_iterations=1)
    assert g.n_correspondences == 8


def test_zero_gate_keeps_exact_hits_and_duplicates(ctx, icp_oracle):
    """max_correspondence_distance 0: only d2 == 0 passes, and the k-NN runs without a cut-off; the source repeats
    some points exactly."""
    T = planes(3, 600)
    hits = np.concatenate([T[:40], T[:40], T[100:120]])  # duplicated exact hits
    S = np.concatenate([hits, T[200:300] + np.float32(0.01)]).astype(np.float32)
    # the fit of exact hits is the identity up to rounding: the thresholds let both fits stop at the first iteration
    g, _ = check(ctx, icp_oracle, T, S, max_correspondence_distance=0.0, max_iterations=3, transformation_epsilon=1e-20,
                 transformation_rotation_epsilon=1 - 1e-12)
    assert (g.state, g.iterations, g.n_correspondences) == (TRANSFORM, 1, 100)


@pytest.mark.parametrize("fit_range", ["zero", "at_d2", "0.05"])
def test_fitness_max_range(ctx, icp_oracle, fit_range):
    T, S, q, t = make_pair(2500)
    q0, t0 = guess_of(q, t)
    if fit_range == "zero":
        rng_v = 0.0
    elif fit_range == "0.05":
        rng_v = 0.05
    else:  # exactly one of the final pass's float d2 (the pose does not depend on the range)
        r = np_icp(T, S, q0, t0, **OPTS)
        _, d2 = nn1(T, transform(r["q"], r["t"], S.astype(np.float64)))
        rng_v = float(np.sort(d2)[len(d2) // 2])
    g, r = check(ctx, icp_oracle, T, S, q0, t0, **dict(OPTS, fitness_max_range=rng_v))
    if fit_range == "zero":
        assert g.fitness == FMAX
    else:
        assert g.fitness < rng_v or (fit_range == "at_d2" and g.fitness <= rng_v)


OPTION_EDGES = {
    "nan_max_corr": dict(max_correspondence_distance=np.nan),
    "nan_fitness_range": dict(fitness_max_range=np.nan),
    "nan_transformation_eps": dict(transformation_epsilon=np.nan, max_iterations=8),
    "nan_rotation_eps": dict(transformation_rotation_epsilon=np.nan, transformation_epsilon=1e-8, max_iterations=60),
    "nan_fitness_eps": dict(euclidean_fitness_epsilon=np.nan, max_iterations=8),
    "negative_max_corr": dict(max_correspondence_distance=-1.0),
    "negative_fitness_range": dict(fitness_max_range=-1.0),
    "negative_rotation_eps": dict(transformation_rotation_epsilon=-0.5, transformation_epsilon=1e-8, max_iterations=60),
    "inf_max_corr": dict(max_correspondence_distance=np.inf),
}


@pytest.mark.parametrize("case", list(OPTION_EDGES))
def test_option_edges(ctx, icp_oracle, case):
    """NaN compares false everywhere: a NaN gate keeps nothing (NO_CORRESPONDENCES at entry), a NaN fitness range gives
    DBL_MAX, NaN epsilons never end the loop, a NaN or non-positive rotation epsilon means 1 - transformation_epsilon.
    Distances are squared, so a negative gate is its absolute value; a negative fitness range keeps nothing."""
    T, S, q, t = make_pair(1500)
    q0, t0 = guess_of(q, t)
    opts = dict(dict(max_iterations=20), **OPTION_EDGES[case])
    g, _ = check(ctx, icp_oracle, T, S, q0, t0, **opts)
    if case == "nan_max_corr":
        assert (g.state, g.iterations) == (NO_CORRESPONDENCES, 0)
    if case in ("nan_fitness_range", "negative_fitness_range"):
        assert g.fitness == FMAX
    if case in ("nan_transformation_eps", "nan_fitness_eps"):
        assert g.state == ITERATIONS and g.iterations == 8
    if case == "negative_max_corr":
        assert bytes(g) == bytes(gpu(ctx, T, S, q0, t0, **dict(opts, max_correspondence_distance=1.0)))
    if case in ("nan_rotation_eps", "negative_rotation_eps"):
        assert bytes(g) == bytes(gpu(ctx, T, S, q0, t0, **dict(opts, transformation_rotation_epsilon=0.0)))


# ---------------------------------------------------------------------------------------------------------------------
# ties and cell sizes
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("iters", [1, 10])
@pytest.mark.parametrize("cell", [0.5, 1.0, 3.0])
def test_ties_on_a_cubic_lattice(ctx, icp_oracle, cell, iters):
    """Source points at edge midpoints, face centres and cube centres of a shuffled unit lattice are equidistant from
    2, 4 or 8 target points (exactly, in float); the lowest target index wins.  The lattice points sit on voxel faces.
    Some target points are repeated at higher indices."""
    T = lattice(6, 1.0, seed=7)
    T = np.concatenate([T, T[::5]])  # duplicates at different indices
    rng = np.random.default_rng(2)
    base = rng.integers(0, 5, (300, 3)).astype(np.float32)
    kind = np.arange(300) % 3
    off = np.where(kind[:, None] == 0, [0.5, 0, 0], np.where(kind[:, None] == 1, [0.5, 0.5, 0], [0.5, 0.5, 0.5]))
    S = (base + off[:, rng.permutation(3)]).astype(np.float32)
    g, _ = check(ctx, icp_oracle, T, S, cell=cell, max_correspondence_distance=1.0, max_iterations=iters)
    if iters == 1:
        assert g.n_correspondences == 300


def test_cell_size_does_not_change_the_result(ctx, icp_oracle):
    T, S, q, t = make_pair(3000)
    q0, t0 = guess_of(q, t)
    res = [gpu(ctx, T, S, q0, t0, cell, **OPTS) for cell in (0.0, 0.25, 1.0, 4.0)]
    w = icp_oracle.icp_align(T, S, q0, t0, **OPTS)
    for g in res:
        same_bytes(g, w)
    agree_ref(res[0], reference(T, S, q0, t0, **OPTS))


# ---------------------------------------------------------------------------------------------------------------------
# geometry
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("yaw", [179.9, 180.0])
def test_rotation_near_half_turn(ctx, icp_oracle, yaw):
    """w ~ 0 and w == 0 in the true rotation and the guess."""
    q_true = quat_z(yaw) if yaw != 180.0 else np.array([0.0, 0.0, 1.0, 0.0])
    T, S, q, t = make_pair(2000, q_true=q_true)
    q0 = q_true if yaw == 180.0 else quat_z(yaw - 0.5)
    g, _ = check(ctx, icp_oracle, T, S, q0, t + [0.1, -0.1, 0.0], **OPTS)
    assert g.converged and rot_dist(g.q, q_true) < 1e-2


def test_kilometres_from_the_origin(ctx, icp_oracle):
    """The scene and the guess at about (2500, -1800, 40) m: the sums about the guess translation keep the
    cross-covariance free of cancellation."""
    far = np.array([2500.25, -1800.5, 40.125])
    T, S, q, t = make_pair(3000)
    T = (T.astype(np.float64) + far).astype(np.float32)
    q0, t0 = guess_of(q, t + far)
    g, _ = check(ctx, icp_oracle, T, S, q0, t0, **OPTS)
    assert g.converged and np.abs(g.tv - (t + far)).max() < 0.05


def test_collinear_source(ctx, icp_oracle):
    """Every source point on one line: the rotation about the line is unobservable, so the transformed points, the
    fitness and the MSE are compared instead of the pose."""
    T = planes(9, 1500)
    d = np.array([0.6, -0.3, 0.2]) / np.linalg.norm([0.6, -0.3, 0.2])
    S = (T[0] + np.linspace(-3, 3, 200)[:, None] * d + [0.05, 0.02, -0.03]).astype(np.float32)
    g, _ = check(ctx, icp_oracle, T, S, points=True, max_correspondence_distance=2.0, max_iterations=4)
    assert g.state == ITERATIONS and np.isfinite(g.q).all() and np.isfinite(g.tv).all()


def test_one_point_target(ctx, icp_oracle):
    """Every correspondence on the same target point: the cross-covariance is exactly zero (power-of-two coordinates,
    64 source points, origin 0), the rotation is the identity and the translation moves the centroid onto the point."""
    T = np.array([[2.0, -4.0, 0.5]], np.float32)
    S = (np.random.default_rng(4).normal(0, 1.0, (64, 3))).astype(np.float32)
    g, r = check(ctx, icp_oracle, T, S, max_iterations=5)
    assert np.isfinite(g.q).all() and np.isfinite(g.tv).all() and np.isfinite(g.fitness) and np.isfinite(g.mse)
    assert np.array_equal(g.q, [0, 0, 0, 1]) and g.n_correspondences == 64
    assert np.abs(g.tv - (T[0] - S.astype(np.float64).mean(0))).max() < 1e-6


# ---------------------------------------------------------------------------------------------------------------------
# non-finite points: never take part (mapOptimization.cpp:151 strips them)
# ---------------------------------------------------------------------------------------------------------------------
BAD = [np.nan, np.inf, -np.inf]


def test_non_finite_target_points(ctx, icp_oracle):
    T, S, q, t = make_pair(2000)
    q0, t0 = guess_of(q, t)
    rng = np.random.default_rng(5)
    at = np.sort(rng.choice(len(T), 60, replace=False))
    Tb = T.copy()
    for k, i in enumerate(at):
        Tb[i, k % 3] = BAD[k % 3]
    g, _ = check(ctx, icp_oracle, Tb, S, q0, t0, **OPTS)
    clean = np.delete(Tb, at, axis=0)  # the finite points keep their order: the same (d2, index) ranking
    assert bytes(g) == bytes(gpu(ctx, clean, S, q0, t0, **OPTS))
    allbad = np.full((50, 3), np.nan, np.float32)
    g, _ = check(ctx, icp_oracle, allbad, S, q0, t0, **OPTS)
    assert (g.state, g.iterations, g.fitness) == (NO_CORRESPONDENCES, 0, FMAX)


def test_non_finite_source_points(ctx, icp_oracle):
    T, S, q, t = make_pair(2000)
    q0, t0 = guess_of(q, t)
    at = np.arange(5, len(S), 37)
    Sb = S.copy()
    for k, i in enumerate(at):
        Sb[i, k % 3] = BAD[k % 3]
    opts = dict(OPTS, fitness_max_range=1.0)
    g, _ = check(ctx, icp_oracle, T, Sb, q0, t0, **opts)
    # the same result as points that sit far outside the gate and the fitness range (the tile layout is unchanged)
    Sf = S.copy()
    Sf[at] = 1e4
    assert bytes(g) == bytes(gpu(ctx, T, Sf, q0, t0, **opts))
    # with no gate and no range at all: a finite point whose transform overflows the float store is non-finite too
    Sb[7] = np.finfo(np.float32).max
    g, _ = check(ctx, icp_oracle, T, Sb, q0, t0, **dict(OPTS, max_correspondence_distance=np.inf, fitness_max_range=np.inf))
    assert np.isfinite(g.fitness) and np.isfinite(g.mse)


# ---------------------------------------------------------------------------------------------------------------------
# entry points and layouts (the C ABI directly)
# ---------------------------------------------------------------------------------------------------------------------
def abi_batch(ctx, maps, src, offs, stride, guesses, dev=False, **opts):
    from ilsm_b200 import binding as b
    n = len(maps)
    hs = (C.c_void_p * n)(*[m._h.value for m in maps])
    res = (b.IcpResult * n)()
    o = b.IcpOpts(**opts)
    offs = np.ascontiguousarray(offs, np.int32)
    g = np.ascontiguousarray(guesses, np.float64).reshape(n, 7)
    fn = ctx._lib.ilsm_icp_align_batch_dev if dev else ctx._lib.ilsm_icp_align_batch
    rc = fn(ctx._h, hs, n, src, offs.ctypes.data, stride, g.ctypes.data, C.byref(o), res)
    assert rc == 0, ctx._lib.ilsm_last_error()
    return [res[i] for i in range(n)]


def three_pairs(ctx):
    out = []
    for k, n in enumerate((700, 2049, 300)):
        T, S, q, t = make_pair(n, seed=20 + k)
        q0, t0 = guess_of(q, t)
        out.append((ctx.new_map().set_input_cloud(T, 1.0), S, np.concatenate([q0, t0])))
    return out


def padded(S, stride, lead):
    """S in records of `stride` bytes after `lead` leading records; every unused word holds garbage, NaN bit patterns
    included."""
    rng = np.random.default_rng(stride)
    words = stride // 4
    a = rng.normal(0, 1e3, (lead + len(S), words)).astype(np.float32)
    a.view(np.uint32)[:, 3::2] = rng.choice(np.array([0x7FC00000, 0xFFFFFFFF, 0x7F800001, 0x7F800000], np.uint32),
                                            a[:, 3::2].shape)
    a[lead:, :3] = S
    return a


@pytest.mark.parametrize("stride", [16, 32])
def test_source_strides_with_garbage_channels(ctx, stride):
    pairs = three_pairs(ctx)
    maps, srcs, guesses = zip(*pairs)
    want = ctx.icp_align_batch(list(maps), list(srcs), [(g[:4], g[4:]) for g in guesses], **OPTS)
    a = padded(np.concatenate(srcs), stride, 0)
    offs = np.concatenate([[0], np.cumsum([len(s) for s in srcs])])
    got = abi_batch(ctx, maps, a.ctypes.data, offs, stride, guesses, **OPTS)
    assert [bytes(r) for r in got] == [bytes(r) for r in want]
    for m in maps:
        m.close()


@pytest.mark.parametrize("stride", [12, 32])
def test_device_entry_point_with_offset_sources(ctx, stride):
    """ilsm_icp_align_batch_dev on torch CUDA memory, the first pair starting at offs[0] > 0."""
    import torch
    pairs = three_pairs(ctx)
    maps, srcs, guesses = zip(*pairs)
    want = ctx.icp_align_batch(list(maps), list(srcs), [(g[:4], g[4:]) for g in guesses], **OPTS)
    lead = 123
    a = padded(np.concatenate(srcs), stride, lead) if stride > 12 else \
        np.concatenate([np.full((lead, 3), np.nan, np.float32), np.concatenate(srcs)])
    d = torch.from_numpy(np.ascontiguousarray(a)).cuda()
    torch.cuda.synchronize()
    offs = lead + np.concatenate([[0], np.cumsum([len(s) for s in srcs])])
    got = abi_batch(ctx, maps, d.data_ptr(), offs, stride, guesses, dev=True, **OPTS)
    assert [bytes(r) for r in got] == [bytes(r) for r in want]
    for m in maps:
        m.close()


# ---------------------------------------------------------------------------------------------------------------------
# batches
# ---------------------------------------------------------------------------------------------------------------------
def test_large_mixed_batch_equals_singles(ilsm, ctx, icp_oracle):
    """About 300 pairs of mixed sizes (more clusters than one wave), empty sources and empty targets among them, in one
    launch: every result equals its single call byte for byte."""
    rng = np.random.default_rng(8)
    scenes = [make_pair(4200, seed=30 + k) for k in range(3)]
    maps = [ctx.new_map().set_input_cloud(T, 1.0) for T, _, _, _ in scenes]
    empty = ctx.new_map().set_input_cloud(np.zeros((0, 3), np.float32))
    targets, sources, guesses = [], [], []
    for p in range(300):
        k = int(rng.integers(0, 3))
        T, S, q, t = scenes[k]
        n = int(rng.choice([0, 1, 2, 5, 100, 256, 257, 1000, 2048, 4200]))
        lo = int(rng.integers(0, len(S) - n + 1))
        targets.append(empty if p % 37 == 5 else maps[k])
        sources.append(S[lo:lo + n])
        guesses.append(guess_of(q, t))
    before = ilsm.launch_count()
    batch = ctx.icp_align_batch(targets, sources, guesses, **OPTS)
    assert ilsm.launch_count() - before == 1
    singles = [ctx.icp_align(m, s, q, t, **OPTS) for m, s, (q, t) in zip(targets, sources, guesses)]
    assert [bytes(r) for r in batch] == [bytes(r) for r in singles]
    assert sum(r.state == NO_CORRESPONDENCES for r in batch) >= sum(len(s) < 3 or m is empty for m, s in zip(targets, sources))
    for p in (0, 1, 2, 5):  # a few against the oracle too
        T = np.zeros((0, 3), np.float32) if targets[p] is empty else scenes[[m for m in maps].index(targets[p])][0]
        same_bytes(batch[p], icp_oracle.icp_align(T, sources[p], *guesses[p], **OPTS))
    for m in maps + [empty]:
        m.close()


def test_rebuilt_target_handle(ctx, icp_oracle):
    """One handle rebuilt with three different clouds (the map alternates its two tables), ICP right after each
    set_input_cloud: the same bytes as a fresh map, and as the oracle."""
    m = ctx.new_map()
    for k, n_tgt in enumerate((1500, 600, 2500)):
        T, S, q, t = make_pair(1800, n_tgt=n_tgt, seed=40 + k)
        q0, t0 = guess_of(q, t)
        g = ctx.icp_align(m.set_input_cloud(T, 1.0), S, q0, t0, **OPTS)
        assert bytes(g) == bytes(gpu(ctx, T, S, q0, t0, **OPTS))
        same_bytes(g, icp_oracle.icp_align(T, S, q0, t0, **OPTS))
    m.close()
