"""Seeded synthetic inputs for the hot path (SURVEY.md section 8d): scene S1 (ground + boxes + poles),
an analytic OS0-64 ray-caster (64 beams +45..-45 deg x 1024 azimuths, organised u*W+v, no-return=(0,0,0)),
map samplers and pose helpers.  Pure numpy; used by tests, bench.py and smoke().  Not an oracle and not a
product kernel -- it only manufactures inputs.
"""
from __future__ import annotations

import numpy as np

SEED_FRAME = 0x5EED0001
SEED_MAP = 0x5EED0002
SEED_GUESS = 0x5EED0003


# ------------------------------------------------------------------------------------------------
# quaternion helpers, Eigen coefficient order (x, y, z, w)
# ------------------------------------------------------------------------------------------------
def quat_mul(a, b):
    ax, ay, az, aw = a
    bx, by, bz, bw = b
    return np.array([aw * bx + ax * bw + ay * bz - az * by, aw * by + ay * bw + az * bx - ax * bz,
                     aw * bz + az * bw + ax * by - ay * bx, aw * bw - ax * bx - ay * by - az * bz])


def quat_from_rotvec(rv):
    rv = np.asarray(rv, np.float64)
    ang = np.linalg.norm(rv)
    if ang < 1e-300:
        return np.array([0.0, 0.0, 0.0, 1.0])
    ax = rv / ang
    return np.concatenate([np.sin(ang / 2) * ax, [np.cos(ang / 2)]])


def quat_to_mat(q):
    x, y, z, w = q / np.linalg.norm(q)
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                     [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                     [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])


def quat_inv(q):
    return np.array([-q[0], -q[1], -q[2], q[3]]) / np.dot(q, q)


def quat_angle(a, b):
    """Rotation angle (rad) between two unit quaternions."""
    d = abs(float(np.dot(a / np.linalg.norm(a), b / np.linalg.norm(b))))
    return 2.0 * np.arccos(min(1.0, d))


# ------------------------------------------------------------------------------------------------
# scene
# ------------------------------------------------------------------------------------------------
class Scene:
    """Ground plane z=0, axis-aligned boxes (buildings) and vertical poles."""

    def __init__(self, seed=SEED_MAP, extent=100.0, n_boxes=40, n_poles=60, corridor=False, length=400.0):
        rng = np.random.default_rng(seed)
        self.extent = float(extent)
        if corridor:
            # scene S2: 3 m x 3 m corridor along +x with pillars every 5 m (SURVEY 8d config 2)
            self.extent = length
            boxes = []
            w = 1.5
            boxes.append([-5.0, w, 0.0, length, w + 1.0, 3.0])     # left wall
            boxes.append([-5.0, -w - 1.0, 0.0, length, -w, 3.0])   # right wall
            boxes.append([-5.0, -w - 1.0, 3.0, length, w + 1.0, 4.0])  # ceiling slab
            for k, x in enumerate(np.arange(2.5, length, 5.0)):
                side = 1 if k % 2 == 0 else -1
                y0, y1 = (w - 0.3, w) if side > 0 else (-w, -w + 0.3)
                boxes.append([x, y0, 0.0, x + 0.4, y1, 3.0])
            self.boxes = np.array(boxes)
            self.poles = np.zeros((0, 5))
            return
        ctr = rng.uniform(-extent * 0.9, extent * 0.9, size=(n_boxes, 2))
        # keep a clearing around the origin where the sensor lives
        ctr = ctr[np.linalg.norm(ctr, axis=1) > 12.0]
        half = rng.uniform(2.0, 8.0, size=(len(ctr), 2))
        h = rng.uniform(3.0, 12.0, size=len(ctr))
        self.boxes = np.column_stack([ctr - half, np.zeros(len(ctr)), ctr + half, h])  # x0 y0 z0 x1 y1 z1
        pc = rng.uniform(-extent * 0.6, extent * 0.6, size=(n_poles, 2))
        pc = pc[np.linalg.norm(pc, axis=1) > 4.0]
        inside = np.zeros(len(pc), bool)
        for b in self.boxes:
            inside |= (pc[:, 0] > b[0] - 0.5) & (pc[:, 0] < b[3] + 0.5) & (pc[:, 1] > b[1] - 0.5) & (pc[:, 1] < b[4] + 0.5)
        pc = pc[~inside]
        self.poles = np.column_stack([pc, np.full(len(pc), 0.12), np.zeros(len(pc)), rng.uniform(3.0, 6.0, len(pc))])

    # -- ray casting ------------------------------------------------------------------------------
    def raycast(self, origin, dirs, max_range=50.0):
        """Nearest hit distance per ray (inf when none) and an object tag:
        0 none, 1 ground, 2 box face, 3 pole, 4 box face within 0.12 m of a vertical box edge."""
        o = np.asarray(origin, np.float64)
        d = np.asarray(dirs, np.float64)
        n = len(d)
        best = np.full(n, np.inf)
        tag = np.zeros(n, np.int8)
        with np.errstate(divide="ignore", invalid="ignore"):
            tg = np.where(d[:, 2] < -1e-9, -o[2] / d[:, 2], np.inf)
        m = tg < best
        best[m], tag[m] = tg[m], 1
        inv = 1.0 / np.where(np.abs(d) < 1e-12, 1e-12, d)
        for b in self.boxes:
            t0 = (b[:3] - o) * inv
            t1 = (b[3:] - o) * inv
            tn = np.minimum(t0, t1).max(axis=1)
            tf = np.maximum(t0, t1).min(axis=1)
            hit = (tn <= tf) & (tn > 1e-6) & (tn < best)
            if hit.any():
                best[hit] = tn[hit]
                hp = o + tn[hit, None] * d[hit]
                ex = np.minimum(np.abs(hp[:, 0] - b[0]), np.abs(hp[:, 0] - b[3]))
                ey = np.minimum(np.abs(hp[:, 1] - b[1]), np.abs(hp[:, 1] - b[4]))
                near_edge = (ex < 0.12) & (ey < 0.12)
                tag[hit] = np.where(near_edge, 4, 2)
        for p in self.poles:
            ox, oy = o[0] - p[0], o[1] - p[1]
            a = d[:, 0] ** 2 + d[:, 1] ** 2
            bq = 2 * (ox * d[:, 0] + oy * d[:, 1])
            c = ox * ox + oy * oy - p[2] ** 2
            disc = bq * bq - 4 * a * c
            with np.errstate(divide="ignore", invalid="ignore"):
                tt = np.where((disc > 0) & (a > 1e-12), (-bq - np.sqrt(np.maximum(disc, 0))) / (2 * a), np.inf)
            z = o[2] + tt * d[:, 2]
            hit = (tt > 1e-6) & (tt < best) & (z >= p[3]) & (z <= p[4])
            best[hit], tag[hit] = tt[hit], 3
        best[best > max_range] = np.inf
        tag[~np.isfinite(best)] = 0
        return best, tag

    # -- map samplers -----------------------------------------------------------------------------
    def sample_map(self, n_total, seed=SEED_MAP, corner_frac=0.12, surf_pitch=0.8, corner_pitch=0.4, jitter=0.05):
        """`n_total` map points (corner array, surf array) sampled on scene structure on jittered lattices.
        Lattice pitches are scaled by a common factor so that the requested count is reached exactly
        (config 3 'S1 densified')."""
        rng = np.random.default_rng(seed)
        n_c = int(round(n_total * corner_frac))
        n_s = n_total - n_c
        surf = self._sample_surf(rng, n_s, surf_pitch, jitter)
        corner = self._sample_corner(rng, n_c, corner_pitch, jitter)
        return corner.astype(np.float32), surf.astype(np.float32)

    def _surf_at(self, pitch):
        E = self.extent
        parts = []
        g = np.arange(-E, E, pitch)
        if len(self.poles) or len(self.boxes) < 10 or True:
            gx, gy = np.meshgrid(g, g, indexing="ij")
            parts.append(np.column_stack([gx.ravel(), gy.ravel(), np.zeros(gx.size)]))
        for b in self.boxes:
            xs = np.arange(b[0], b[3], pitch)
            ys = np.arange(b[1], b[4], pitch)
            zs = np.arange(b[2] + pitch / 2, b[5], pitch)
            for yv in (b[1], b[4]):
                X, Z = np.meshgrid(xs, zs, indexing="ij")
                parts.append(np.column_stack([X.ravel(), np.full(X.size, yv), Z.ravel()]))
            for xv in (b[0], b[3]):
                Y, Z = np.meshgrid(ys, zs, indexing="ij")
                parts.append(np.column_stack([np.full(Y.size, xv), Y.ravel(), Z.ravel()]))
        return np.concatenate(parts)

    def _corner_at(self, pitch):
        parts = []
        for b in self.boxes:
            zs = np.arange(b[2] + pitch / 2, b[5], pitch)
            for xv in (b[0], b[3]):
                for yv in (b[1], b[4]):
                    parts.append(np.column_stack([np.full(len(zs), xv), np.full(len(zs), yv), zs]))
        for p in self.poles:
            zs = np.arange(p[3] + pitch / 2, p[4], pitch)
            parts.append(np.column_stack([np.full(len(zs), p[0]), np.full(len(zs), p[1]), zs]))
        return np.concatenate(parts) if parts else np.zeros((0, 3))

    @staticmethod
    def _fit_count(fn, n, pitch0):
        """Shrink the pitch until fn(pitch) yields >= n points."""
        pitch = pitch0
        pts = fn(pitch)
        it = 0
        while len(pts) < n and it < 40:
            pitch *= max(0.5, (len(pts) / max(n, 1)) ** 0.5 * 0.97)
            pts = fn(pitch)
            it += 1
        return pts

    def _sample_surf(self, rng, n, pitch, jitter):
        pts = self._fit_count(self._surf_at, n, pitch)
        sel = rng.permutation(len(pts))[:n]
        sel.sort()
        return pts[sel] + rng.uniform(-jitter, jitter, size=(n, 3))

    def _sample_corner(self, rng, n, pitch, jitter):
        pts = self._fit_count(self._corner_at, n, pitch)
        sel = rng.permutation(len(pts))[:n]
        sel.sort()
        return pts[sel] + rng.uniform(-jitter, jitter, size=(n, 3))


# ------------------------------------------------------------------------------------------------
# sensor
# ------------------------------------------------------------------------------------------------
def os0_dirs(H=64, W=1024, fov_deg=45.0):
    """Unit ray directions of an OS0-64 in the sensor frame, organised row-major u*W+v (u = beam)."""
    elev = np.deg2rad(np.linspace(fov_deg, -fov_deg, H))
    az = -2.0 * np.pi * np.arange(W) / W  # Ouster spins clockwise seen from above
    ce, se = np.cos(elev)[:, None], np.sin(elev)[:, None]
    d = np.stack([ce * np.cos(az)[None, :], ce * np.sin(az)[None, :], np.broadcast_to(se, (H, W))], axis=-1)
    return d.reshape(-1, 3)


def make_frame(scene, q_ws, t_ws, seed=SEED_FRAME, H=64, W=1024, noise=0.01, max_range=50.0, stride_floats=4, fov_deg=45.0):
    """Organised H*W cloud in the SENSOR frame: float32 rows [x y z intensity] (or PCL 8-float PointXYZI when
    stride_floats=8: x y z pad intensity pad pad pad).  Returns (cloud, tag)."""
    rng = np.random.default_rng(seed)
    d_s = os0_dirs(H, W, fov_deg)
    R = quat_to_mat(np.asarray(q_ws, np.float64))
    rng_, tag = scene.raycast(np.asarray(t_ws, np.float64), d_s @ R.T, max_range)
    r = rng_ + rng.normal(0.0, noise, size=len(rng_))
    ok = np.isfinite(rng_)
    pts = np.where(ok[:, None], d_s * np.where(ok, r, 0.0)[:, None], 0.0)
    inten = np.where(ok, rng.uniform(0.0, 255.0, size=len(r)), 0.0)
    cloud = np.zeros((H * W, stride_floats), np.float32)
    cloud[:, :3] = pts
    cloud[:, 3 if stride_floats == 4 else 4] = inten
    return cloud, tag


def make_frames_torch(scene, poses, seed0, device, H=64, W=1024, noise=0.01, max_range=50.0, fov_deg=45.0, out=None):
    """The same sensor model as make_frame for a whole sequence, ray-cast on the GPU with torch (data generation only:
    a 2000-frame sequence takes seconds instead of half an hour with the numpy ray-caster).  poses: [(q_ws, t_ws)];
    frame k uses torch seed seed0 + k for the range noise and the intensities.  Returns a pinned (F, H*W, 4) float32
    host tensor of organised sensor-frame clouds (x y z intensity; no-return = 0).  Boxes further than max_range from the
    sensor are culled per frame; poles are handled like Scene.raycast.  Not bit-identical to make_frame (float64 on the
    GPU, another noise stream) -- both the CUDA path and the oracle consume the arrays it returns."""
    import torch
    F = len(poses)
    if out is None:
        out = torch.empty((F, H * W, 4), dtype=torch.float32).pin_memory()
    d_s = torch.from_numpy(os0_dirs(H, W, fov_deg)).to(device)
    boxes = torch.from_numpy(np.asarray(scene.boxes, np.float64).reshape(-1, 6)).to(device)
    poles = torch.from_numpy(np.asarray(scene.poles, np.float64).reshape(-1, 5)).to(device)
    inf = float("inf")
    gen = torch.Generator(device=device)
    for k, (q, t) in enumerate(poses):
        R = torch.from_numpy(quat_to_mat(np.asarray(q, np.float64))).to(device)
        o = torch.from_numpy(np.asarray(t, np.float64)).to(device)
        d = d_s @ R.T
        best = torch.where(d[:, 2] < -1e-9, -o[2] / d[:, 2], torch.full_like(d[:, 2], inf))
        inv = 1.0 / torch.where(d.abs() < 1e-12, torch.full_like(d, 1e-12), d)
        if len(boxes):
            # cull by the box's distance to the sensor in the xy plane
            cx = torch.clamp(o[0], boxes[:, 0], boxes[:, 3]) - o[0]
            cy = torch.clamp(o[1], boxes[:, 1], boxes[:, 4]) - o[1]
            near = boxes[(cx * cx + cy * cy) <= (max_range + 1.0) ** 2]
            if len(near):
                t0 = (near[None, :, :3] - o) * inv[:, None, :]
                t1 = (near[None, :, 3:] - o) * inv[:, None, :]
                tn = torch.minimum(t0, t1).amax(dim=2)
                tf = torch.maximum(t0, t1).amin(dim=2)
                hit = (tn <= tf) & (tn > 1e-6)
                best = torch.minimum(best, torch.where(hit, tn, torch.full_like(tn, inf)).amin(dim=1))
        if len(poles):
            ox, oy = o[0] - poles[None, :, 0], o[1] - poles[None, :, 1]
            a = (d[:, 0] ** 2 + d[:, 1] ** 2)[:, None]
            bq = 2 * (ox * d[:, 0:1] + oy * d[:, 1:2])
            cq = ox * ox + oy * oy - poles[None, :, 2] ** 2
            disc = bq * bq - 4 * a * cq
            tt = torch.where((disc > 0) & (a > 1e-12), (-bq - torch.sqrt(disc.clamp_min(0))) / (2 * a), torch.full_like(disc, inf))
            z = o[2] + tt * d[:, 2:3]
            ok = (tt > 1e-6) & (z >= poles[None, :, 3]) & (z <= poles[None, :, 4])
            best = torch.minimum(best, torch.where(ok, tt, torch.full_like(tt, inf)).amin(dim=1))
        ok = torch.isfinite(best) & (best <= max_range)
        gen.manual_seed(int(seed0) + k)
        r = best + noise * torch.randn(len(best), generator=gen, device=device, dtype=torch.float64)
        inten = 255.0 * torch.rand(len(best), generator=gen, device=device, dtype=torch.float64)
        r = torch.where(ok, r, torch.zeros_like(r))
        cloud = torch.zeros((H * W, 4), dtype=torch.float32, device=device)
        cloud[:, :3] = (d_s * r[:, None]).to(torch.float32)
        cloud[:, 3] = torch.where(ok, inten, torch.zeros_like(inten)).to(torch.float32)
        out[k].copy_(cloud, non_blocking=True)
    torch.cuda.synchronize(device)
    return out


def corridor_poses(n_frames, step=0.2):
    """SURVEY 8d config 2 trajectory: `step` m per frame forward along the corridor, sinusoidal yaw +-5 degrees."""
    poses = []
    for k in range(n_frames):
        yaw = np.deg2rad(5.0) * np.sin(2 * np.pi * k / 50.0)
        poses.append((quat_from_rotvec([0.0, 0.0, yaw]), np.array([2.0 + step * k, 0.1 * np.sin(k / 15.0), 1.2])))
    return poses


def voxel_centroid_np(pts, leaf):
    """Plain numpy voxel-centroid thinning used only to synthesise feature stacks (NOT the PCL restatement)."""
    if len(pts) == 0:
        return pts
    key = np.floor(pts[:, :3] / leaf).astype(np.int64)
    key -= key.min(axis=0)
    dims = key.max(axis=0) + 1
    lin = key[:, 0] + dims[0] * (key[:, 1] + dims[1] * key[:, 2])
    uniq, inv = np.unique(lin, return_inverse=True)
    out = np.zeros((len(uniq), pts.shape[1]), np.float64)
    np.add.at(out, inv, pts.astype(np.float64))
    out /= np.bincount(inv)[:, None]
    return out.astype(np.float32)


def synth_stacks(cloud, tag, line_res=0.4, plane_res=0.8):
    """Feature stacks straight from ray-cast tags (poles / box edges -> corner, everything else -> surf),
    thinned like laserMapping.cpp:608-616.  Stand-in for the front end when only the registration is run."""
    xyz = cloud[:, :3]
    valid = tag > 0
    corner = xyz[valid & ((tag == 3) | (tag == 4))]
    surf = xyz[valid & ((tag == 1) | (tag == 2))]
    c = voxel_centroid_np(corner, line_res)
    s = voxel_centroid_np(surf, plane_res)
    c4 = np.zeros((len(c), 4), np.float32)
    s4 = np.zeros((len(s), 4), np.float32)
    c4[:, :3], s4[:, :3] = c, s
    return c4, s4


def default_pose():
    """Ground-truth sensor pose T* for config 1."""
    q = quat_from_rotvec([0.01, -0.015, 0.3])
    t = np.array([0.5, -0.3, 1.5])
    return q, t


def perturb_pose(q, t, seed=SEED_GUESS, dt=0.2, drot_deg=2.0):
    rng = np.random.default_rng(seed)
    dq = quat_from_rotvec(np.deg2rad(rng.uniform(-drot_deg, drot_deg, 3)))
    return quat_mul(q, dq), t + rng.uniform(-dt, dt, 3)


def config1(n_map=100_000, seed_shift=0):
    """BASELINE config 1: one OS0-64 frame + 100k-point map + perturbed initial guess."""
    # below 100k points the scene shrinks (same lattice pitch); above, the 100 m scene is densified (config 3)
    frac = min(1.0, n_map / 100_000.0)
    scene = Scene(SEED_MAP + seed_shift, extent=max(25.0, 100.0 * frac ** 0.5), n_boxes=max(6, int(40 * frac)),
                  n_poles=max(8, int(60 * frac)))
    map_corner, map_surf = scene.sample_map(n_map, SEED_MAP + seed_shift)
    q, t = default_pose()
    cloud, tag = make_frame(scene, q, t, SEED_FRAME + seed_shift)
    corner, surf = synth_stacks(cloud, tag)
    q0, t0 = perturb_pose(q, t, SEED_GUESS + seed_shift)
    return dict(scene=scene, map_corner=map_corner, map_surf=map_surf, cloud=cloud, tag=tag, corner=corner,
                surf=surf, q_true=q, t_true=t, q0=q0, t0=t0)


# ------------------------------------------------------------------------------------------------
# ScanContext database (SURVEY 8d config 5)
# ------------------------------------------------------------------------------------------------
SEED_SC = 0x5EED0200


def sc_database(n, seed=SEED_SC):
    """n synthetic 20x60 descriptors: each bin empty (0) w.p. 0.4, else a max-height value U(0,6) m; float32."""
    rng = np.random.default_rng(seed)
    d = rng.uniform(0.0, 6.0, size=(n, 20, 60)).astype(np.float32)
    d[rng.random((n, 20, 60)) < 0.4] = 0.0
    return d


SC_CHUNK = 1000


def sc_database_chunk(ci, n_total):
    """Chunk ci (SC_CHUNK keyframes, seeded by its index) of a database of n_total keyframes: every rank of a sharded run
    generates its own shard -- and the source entries of the queries -- without materialising the whole database."""
    return sc_database(min(SC_CHUNK, n_total - ci * SC_CHUNK), seed=SEED_SC + 17 * ci)


def sc_database_range(lo, hi, n_total):
    """Descriptors [lo, hi) of the chunk-seeded database."""
    parts = []
    for ci in range(lo // SC_CHUNK, (hi + SC_CHUNK - 1) // SC_CHUNK):
        c = sc_database_chunk(ci, n_total)
        parts.append(c[max(lo, ci * SC_CHUNK) - ci * SC_CHUNK: min(hi, (ci + 1) * SC_CHUNK) - ci * SC_CHUNK])
    return np.concatenate(parts) if parts else np.zeros((0, 20, 60), np.float32)


def sc_chunked_queries(n_total, n_q, seed=SEED_SC + 1, noise=0.05, exclude_recent=50):
    """n_q queries against the chunk-seeded database: entries older than the newest `exclude_recent` re-rendered with a
    known yaw shift + noise (SURVEY 8d config 5).  Returns (queries (n_q, 20, 60), true ids, true shifts)."""
    rng = np.random.default_rng(seed)
    ids = np.sort(rng.integers(0, n_total - exclude_recent, n_q))  # sorted: consecutive queries share source chunks
    shifts = rng.integers(0, 60, n_q)
    q = np.empty((n_q, 20, 60), np.float32)
    cache = (-1, None)
    for j, (i, s) in enumerate(zip(ids, shifts)):
        ci = int(i) // SC_CHUNK
        if cache[0] != ci:
            cache = (ci, sc_database_chunk(ci, n_total))
        d = np.roll(cache[1][int(i) - ci * SC_CHUNK], int(s), axis=1).astype(np.float32)
        q[j] = d + rng.normal(0.0, noise, d.shape).astype(np.float32) * (d != 0)
    return q, ids.astype(np.int32), shifts.astype(np.int32)


def sc_queries(db, n_q, seed=SEED_SC + 1, noise=0.05):
    """Queries = database entries re-rendered with a yaw shift of U{0..59} sectors plus N(0, noise) on the occupied
    bins, so the true id and shift are known.  Returns (queries, true ids, true shifts)."""
    rng = np.random.default_rng(seed)
    ids = rng.integers(0, len(db), n_q)
    shifts = rng.integers(0, 60, n_q)
    q = np.empty((n_q, 20, 60), np.float32)
    for j, (i, s) in enumerate(zip(ids, shifts)):
        d = np.roll(db[i], int(s), axis=1).astype(np.float32)  # == circshift(candidate, s) (Scancontext.cpp:44-68)
        occ = d != 0
        d = d + (rng.normal(0.0, noise, d.shape).astype(np.float32) * occ)
        q[j] = d
    return q, ids.astype(np.int32), shifts.astype(np.int32)


def loop_keyframes(n_per_lap=12, laps=2, radius=8.0, leaf=0.4, seed=0x5EED1C00, scene=None):
    """Keyframes of a closed path through the box scene (Scene()): `laps` times around a circle of `radius` m, every lap
    0.1 m further out and 3 degrees more yaw than the one before, so that keyframe k of a lap revisits keyframe k of the
    first.  Per keyframe: true pose (q, t), `src` = its OS0-64 frame thinned by VoxelGrid(leaf) in the sensor frame,
    `world` = the same points in the world frame.  Loop-closure verification workload (tools/icp_bench.py, ICP tests)."""
    scene = scene or Scene()
    out = []
    for lap in range(laps):
        for k in range(n_per_lap):
            a = 2 * np.pi * k / n_per_lap
            r = radius + 0.1 * lap
            q = quat_from_rotvec([0.0, 0.0, a + np.pi / 2 + np.deg2rad(3.0 * lap)])
            t = np.array([r * np.cos(a), r * np.sin(a), 1.5])
            cloud, _ = make_frame(scene, q, t, seed=seed + lap * n_per_lap + k)
            pts = cloud[np.any(cloud[:, :3] != 0, axis=1), :3]
            src = voxel_centroid_np(pts, leaf)
            world = (src.astype(np.float64) @ quat_to_mat(q).T + t).astype(np.float32)
            out.append(dict(q=q, t=t, src=src, world=world, lap=lap, k=k))
    return out


def loop_submap(kfs, c, n_per_lap, half=2, leaf=0.4):
    """World-frame submap around keyframe c: keyframes c-half .. c+half of c's lap (cyclic), VoxelGrid(leaf)."""
    lap0 = (c // n_per_lap) * n_per_lap
    ids = [lap0 + (c - lap0 + d) % n_per_lap for d in range(-half, half + 1)]
    return voxel_centroid_np(np.concatenate([kfs[i]["world"] for i in ids]), leaf)
