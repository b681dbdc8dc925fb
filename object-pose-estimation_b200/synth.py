"""Synthetic inputs for tests and benchmarks (SURVEY section 8d; master seed 20261018).

Nothing here reads /root/reference: the model is a procedural "drill-like" solid (body cylinder, handle
box, chuck cone) area-sampled to the bundled model's size (157 825 points, bbox about 0.2 x 0.2 x 0.09 m,
centred on the origin like D&L/3DModel/drillNewModelOrigin.pcd), the scenes are z-buffered 640x480
Kinect-like depth images with the intrinsics of D&L/src/datagrabber.cpp:146-150 (fx = fy = 525,
cx = 319.5, cy = 239.5, depth in uint16 millimetres, Z == 0 or Z > 2 m dropped as in :34).
"""
import numpy as np

MASTER_SEED = 20261018
FX = FY = 525.0
CX, CY = 319.5, 239.5
W, H = 640, 480


def rng_for(frame, stream=0):
    return np.random.default_rng([MASTER_SEED, int(stream), int(frame)])


# ------------------------------------------------------------------------------------------- model ----
def _sample_cylinder(rng, n, r, h, axis_z0):
    """lateral surface + two caps of a z-aligned cylinder, area-weighted."""
    a_side, a_cap = 2 * np.pi * r * h, np.pi * r * r
    k = rng.choice(3, size=n, p=np.array([a_side, a_cap, a_cap]) / (a_side + 2 * a_cap))
    th = rng.uniform(0, 2 * np.pi, n)
    rr = r * np.sqrt(rng.uniform(0, 1, n))
    z = rng.uniform(0, h, n)
    x = np.where(k == 0, r * np.cos(th), rr * np.cos(th))
    y = np.where(k == 0, r * np.sin(th), rr * np.sin(th))
    z = np.where(k == 0, z, np.where(k == 1, 0.0, h)) + axis_z0
    return np.stack([x, y, z], 1)


def _sample_box(rng, n, lo, hi):
    lo, hi = np.asarray(lo, float), np.asarray(hi, float)
    d = hi - lo
    areas = np.array([d[1] * d[2], d[1] * d[2], d[0] * d[2], d[0] * d[2], d[0] * d[1], d[0] * d[1]])
    face = rng.choice(6, size=n, p=areas / areas.sum())
    p = lo + rng.uniform(0, 1, (n, 3)) * d
    ax = face // 2
    side = face % 2
    p[np.arange(n), ax] = np.where(side == 0, lo[ax], hi[ax])
    return p


def _sample_cone(rng, n, r0, r1, h, z0):
    """frustum lateral surface, radius r0 at z0 -> r1 at z0+h (area-weighted along the slant)."""
    u = rng.uniform(0, 1, n)
    # area density proportional to radius: invert CDF of r(t) = r0 + (r1-r0) t
    if abs(r1 - r0) < 1e-12:
        t = u
    else:
        t = (np.sqrt(r0 * r0 + u * (r1 * r1 - r0 * r0)) - r0) / (r1 - r0)
    r = r0 + (r1 - r0) * t
    th = rng.uniform(0, 2 * np.pi, n)
    return np.stack([r * np.cos(th), r * np.sin(th), z0 + h * t], 1)


def make_model(n_points=157825, seed=0):
    """Procedural drill-like object, float32 (n,3), centred on the origin."""
    rng = rng_for(seed, stream=1)
    parts = [
        ("body", lambda m: _sample_cylinder(rng, m, 0.032, 0.13, -0.065), 2 * np.pi * 0.032 * 0.13 + 2 * np.pi * 0.032 ** 2),
        ("chuck", lambda m: _sample_cone(rng, m, 0.032, 0.012, 0.045, 0.065), np.pi * (0.032 + 0.012) * 0.05),
        ("bit", lambda m: _sample_cylinder(rng, m, 0.004, 0.03, 0.110), 2 * np.pi * 0.004 * 0.03),
        ("handle", lambda m: _sample_box(rng, m, (-0.02, -0.16, -0.05), (0.02, -0.03, -0.005)), 2 * (0.04 * 0.13 + 0.04 * 0.045 + 0.13 * 0.045)),
        ("battery", lambda m: _sample_box(rng, m, (-0.035, -0.19, -0.075), (0.035, -0.16, 0.02)), 2 * (0.07 * 0.03 + 0.07 * 0.095 + 0.03 * 0.095)),
    ]
    areas = np.array([a for _, _, a in parts])
    counts = np.floor(n_points * areas / areas.sum()).astype(int)
    counts[0] += n_points - counts.sum()
    pts = np.concatenate([f(c) for (_, f, _), c in zip(parts, counts)], 0)
    # z is the tool axis; rotate so the bbox is roughly 0.2 x 0.2 x 0.09 (x: tool axis, y: handle, z: thickness)
    pts = pts[:, [2, 1, 0]]
    pts -= 0.5 * (pts.min(0) + pts.max(0))
    rng.shuffle(pts, axis=0)
    return np.ascontiguousarray(pts, dtype=np.float32)


def bundled_model(with_rgb=False):
    """The model cloud the reference ships (D&L/3DModel/drillNewModelOrigin.pcd, 157 825 points; BASELINE.json configs[0]),
    from the committed fixture tests/golden/drill_model.npz (made by tests/golden/make_model_fixture.py)."""
    import os
    path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "drill_model.npz")
    z = np.load(path)
    xyz = np.ascontiguousarray(z["xyz"], np.float32)
    return (xyz, z["rgb"]) if with_rgb else xyz


# ------------------------------------------------------------------------------------------- poses ----
def random_rotation(rng):
    q = rng.normal(size=4)
    q /= np.linalg.norm(q)
    w, x, y, z = q
    return np.array([
        [1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
        [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
        [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])


def rotation_about(axis, angle):
    axis = np.asarray(axis, float)
    axis = axis / np.linalg.norm(axis)
    K = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    return np.eye(3) + np.sin(angle) * K + (1 - np.cos(angle)) * (K @ K)


def random_pose(rng, z_range=(0.6, 1.6), xy=0.2):
    T = np.eye(4)
    T[:3, :3] = random_rotation(rng)
    T[:3, 3] = [rng.uniform(-xy, xy), rng.uniform(-xy, xy), rng.uniform(*z_range)]
    return T


def small_pose(rng, max_deg=10.0, max_t=0.02):
    ax = rng.normal(size=3)
    T = np.eye(4)
    T[:3, :3] = rotation_about(ax, np.deg2rad(rng.uniform(0.3 * max_deg, max_deg)))
    t = rng.normal(size=3)
    T[:3, 3] = t / np.linalg.norm(t) * rng.uniform(0.3 * max_t, max_t)
    return T


def apply(T, pts):
    return (pts.astype(np.float64) @ T[:3, :3].T + T[:3, 3]).astype(np.float32)


def pose_error(Ta, Tb):
    """(rotation angle in rad, translation distance in m) between two 4x4 poses."""
    Ra, Rb = np.asarray(Ta, float)[:3, :3], np.asarray(Tb, float)[:3, :3]
    # ||Ra - Rb||_F = 2*sqrt(2)*sin(angle/2): well conditioned for tiny angles (arccos of the trace is not)
    s = np.linalg.norm(Ra - Rb) / (2.0 * np.sqrt(2.0))
    return float(2.0 * np.arcsin(np.clip(s, 0, 1))), float(np.linalg.norm(np.asarray(Ta, float)[:3, 3] - np.asarray(Tb, float)[:3, 3]))


# ------------------------------------------------------------------------------------------ scenes ----
def render_scene(model, pose, rng, outlier_frac=0.0, hand=False, wall_z=1.6, noise=True):
    """Z-buffer the posed model, a table plane under it and a back wall into a 640x480 depth image.

    Returns (cloud (480,640,3) float32 with NaN for invalid pixels, object mask (480,640) bool).
    """
    P = apply(pose, model).astype(np.float64)
    depth = np.full((H, W), np.inf)
    u = np.rint(P[:, 0] * FX / P[:, 2] + CX).astype(int)
    v = np.rint(P[:, 1] * FY / P[:, 2] + CY).astype(int)
    ok = (P[:, 2] > 0.1) & (u >= 0) & (u < W) & (v >= 0) & (v < H)
    np.minimum.at(depth, (v[ok], u[ok]), P[ok, 2])
    obj = np.isfinite(depth)
    # table: plane through the lowest object point along the camera's "down" direction, tilted 30 deg
    n = np.array([0.0, -np.cos(np.deg2rad(30.0)), -np.sin(np.deg2rad(30.0))])  # plane normal (pointing up/toward camera)
    d = (P @ n).min() - 0.002
    uu, vv = np.meshgrid(np.arange(W), np.arange(H))
    ray = np.stack([(uu - CX) / FX, (vv - CY) / FY, np.ones_like(uu, float)], -1)
    denom = ray @ n
    with np.errstate(divide="ignore", invalid="ignore"):
        zt = np.where(denom < -1e-9, d / denom, np.inf)
    zt = np.where(zt > 0.1, zt, np.inf)
    bg = np.minimum(zt, wall_z)
    depth = np.where(obj & (depth <= bg), depth, bg)
    obj &= depth < bg
    if hand:
        # a capsule between camera and object hiding 20-40 % of the object's pixels
        ys, xs = np.nonzero(obj)
        if len(xs):
            frac = rng.uniform(0.2, 0.4)
            cx0 = np.quantile(xs, frac)
            hide = obj & (uu <= cx0)
            zc = np.nanmin(np.where(obj, depth, np.nan)) - 0.08
            depth = np.where(hide, zc + 0.01 * np.sin(vv / 7.0), depth)
            obj &= ~hide
    if noise:
        depth = depth + rng.normal(size=depth.shape) * 0.0015 * depth * depth
    if outlier_frac > 0:
        m = rng.uniform(size=depth.shape) < outlier_frac
        depth = np.where(m, rng.uniform(0.4, 2.0, size=depth.shape), depth)
        obj &= ~m
    mm = np.rint(depth * 1000.0)
    mm = np.where((mm <= 0) | (mm > 2000), 0, mm).astype(np.uint16)  # datagrabber.cpp:34 — Z == 0 or Z > 2 m dropped
    z = mm.astype(np.float32) * np.float32(0.001)
    cloud = np.stack([(uu - CX).astype(np.float32) * z / np.float32(FX), (vv - CY).astype(np.float32) * z / np.float32(FY), z], -1)
    cloud[mm == 0] = np.nan
    return cloud.astype(np.float32), obj & (mm > 0)


def cluster_from_scene(cloud, obj_mask, rim_px=3):
    """What the reference feeds estimateFinalPose (D&L/src/rosinterface.cpp:246-250): the segmented object
    cluster — here the analytically known object pixels plus a thin rim of neighbouring table pixels."""
    from scipy.ndimage import binary_dilation
    m = binary_dilation(obj_mask, iterations=rim_px) if rim_px > 0 else obj_mask
    pts = cloud[m]
    pts = pts[np.isfinite(pts).all(1)]
    return np.ascontiguousarray(pts, np.float32)


def make_frame(model, frame, outlier_frac=0.0, hand=False, z_range=(0.6, 1.6)):
    """C1/C5 frame `frame`: (cluster points, organised cloud, ground-truth pose)."""
    rng = rng_for(frame, stream=2)
    pose = random_pose(rng, z_range=z_range)
    cloud, mask = render_scene(model, pose, rng, outlier_frac=outlier_frac, hand=hand)
    return cluster_from_scene(cloud, mask), cloud, pose


def make_sequence(model, seq, n_frames, max_deg=10.0, max_t=0.02):
    """A tracking sequence: per frame (cluster points, organised cloud, pose), the pose random at frame 0 and then composed with
    small_pose steps."""
    rng = rng_for(seq, stream=5)
    pose = random_pose(rng)
    out = []
    for _ in range(n_frames):
        cloud, mask = render_scene(model, pose, rng)
        out.append((cluster_from_scene(cloud, mask), cloud, pose))
        pose = small_pose(rng, max_deg, max_t) @ pose
    return out


TABLE_UP = np.array([0.0, -np.cos(np.deg2rad(30.0)), -np.sin(np.deg2rad(30.0))])   # render_scene's table normal
TABLE_AWAY = np.array([0.0, -np.sin(np.deg2rad(30.0)), np.cos(np.deg2rad(30.0))])  # in the table plane, away from the camera


def make_scene_sequence(model, seq, n_frames, distractors=2, jump_at=None, max_deg=5.0, max_t=0.01):
    """A multi-object tracking sequence in depth images: the object on the table in front of the camera, turned and moved by a
    small_pose step (about its own centre) per frame, next to `distractors` (0, 1 or 2) static objects on the same table at least
    10 cm away from it: a cylinder larger than the object (its cluster is the largest, rank 0) and a small box. At frame jump_at
    the object moves 12 cm further along the table. Returns (depth (n_frames, 480, 640) uint16 millimetres, object poses)."""
    rng = rng_for(seq, stream=6)
    R = random_rotation(rng)
    # x = -0.12 at z = 1: the middle of the crop, whose x is the image column measured from cy (depth_to_cloud's row/column quirk)
    t = np.array([rng.uniform(-0.16, -0.08), 0.0, rng.uniform(0.95, 1.05)])
    # the object's centre sits half its extent above the table; distractors stand on the same level, to its left and right
    base = t - TABLE_UP * 0.05
    still = []
    if distractors >= 1:
        cyl = _sample_cylinder(rng, 60000, 0.07, 0.22, 0.0)                # axis along the table normal, foot on the table
        frame = np.stack([np.array([1.0, 0.0, 0.0]), TABLE_AWAY, TABLE_UP], 1)
        still.append(cyl @ frame.T + base + np.array([0.30, 0.0, 0.0]) - TABLE_UP * 0.01)
    if distractors >= 2:
        box = _sample_box(rng, 20000, (-0.03, -0.03, 0.0), (0.03, 0.03, 0.06))
        frame = np.stack([np.array([1.0, 0.0, 0.0]), TABLE_AWAY, TABLE_UP], 1)
        still.append(box @ frame.T + base + np.array([-0.27, 0.0, 0.0]) - TABLE_UP * 0.01)
    depth, poses = [], []
    for k in range(n_frames):
        if k == jump_at:
            t = t + 0.12 * TABLE_AWAY
        pose = np.eye(4)
        pose[:3, :3], pose[:3, 3] = R, t
        pts = np.concatenate([apply(pose, model)] + [p.astype(np.float32) for p in still], 0)
        cloud, _ = render_scene(pts, np.eye(4), rng)
        depth.append(np.rint(np.nan_to_num(cloud[..., 2], nan=0.0).astype(np.float64) * 1000.0).astype(np.uint16))
        poses.append(pose)
        step = small_pose(rng, max_deg, max_t)
        R, t = step[:3, :3] @ R, t + step[:3, 3]
    return np.stack(depth), poses


def icp_pair(n=50000, seed=0, model=None, max_deg=10.0, max_t=0.02, sigma=0.001, outlier_frac=0.10):
    """C2: target = n model-surface points, source = an independent n-sample under a small perturbation,
    sigma = 1 mm noise, 10 % of the source replaced by outliers in the (inflated) bounding box."""
    rng = rng_for(seed, stream=3)
    if model is None:
        model = make_model()
    it = rng.choice(len(model), size=n, replace=len(model) < n)
    is_ = rng.choice(len(model), size=n, replace=len(model) < n)
    tgt = model[it].astype(np.float32)
    T = small_pose(rng, max_deg, max_t)
    src = apply(np.linalg.inv(T), model[is_]) + rng.normal(size=(n, 3)).astype(np.float32) * np.float32(sigma)
    k = int(outlier_frac * n)
    if k:
        lo, hi = model.min(0) - 0.05, model.max(0) + 0.05
        src[rng.choice(n, size=k, replace=False)] = rng.uniform(lo, hi, size=(k, 3)).astype(np.float32)
    return np.ascontiguousarray(src, np.float32), np.ascontiguousarray(tgt, np.float32), T


def turntable_views(model, n_views=36, z=0.8, seed=0, first=None):
    """C4: n_views object-only views at 360/n_views degree steps, each in its own camera frame (`first`: render only
    the first that many)."""
    out = []
    for i in range(n_views if first is None else min(first, n_views)):
        rng = rng_for(seed * 1000 + i, stream=4)
        T = np.eye(4)
        T[:3, :3] = rotation_about([0, 1, 0], 2 * np.pi * i / n_views) @ rotation_about([1, 0, 0], np.deg2rad(-60))
        T[:3, 3] = [0, 0, z]
        cloud, mask = render_scene(model, T, rng)
        pts = cloud[mask]
        out.append((np.ascontiguousarray(pts[np.isfinite(pts).all(1)], np.float32), T))
    return out
