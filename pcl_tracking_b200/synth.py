"""Synthetic Kinect2-shaped clouds (SURVEY.md section 8d).

An organised 512x424 depth image (fx=fy=365, cx=256, cy=212) is ray-cast from a tilted table
plane, a back wall and K moving objects (oriented boxes / spheres, saturated colours), with
depth noise sigma = 1.5 mm * z^2 and 5 % NaN holes.  Points are the 16-byte packed layout
{x, y, z, rgba(b,g,r,a)}; the reference's sensor topic is /kinect2/{sd,qhd}/points
(ref: src/auto_tracking.cpp:775-776).  numpy only: this is input generation, not the hot path.
"""
import numpy as np

POINT = np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("rgba", "<u4")])

KINECT2_SD = dict(width=512, height=424, f=365.0, cx=256.0, cy=212.0)
KINECT2_QHD = dict(width=960, height=540, f=540.0, cx=480.0, cy=270.0)

_TABLE_N = np.array([0.0, -0.766044443, -0.64278761])  # ~50 deg tilt (cf. ref: camera_robot_calibrationtxt:4)
_TABLE_P = np.array([0.0, 0.30, 1.20])


def _rot(axis, angle):
    axis = np.asarray(axis, dtype=np.float64)
    axis = axis / np.linalg.norm(axis)
    K = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    return np.eye(3) + np.sin(angle) * K + (1 - np.cos(angle)) * (K @ K)


def table_frame():
    """Orthonormal basis (u, v, n) of the table plane; objects are placed at P + a*u + b*v + h*n."""
    n = _TABLE_N.copy()
    u = np.array([1.0, 0.0, 0.0])
    v = np.cross(n, u)
    v /= np.linalg.norm(v)
    return u, v, n


def default_objects(k=1, seed=7):
    """K objects resting on the table.  Each: dict(kind, centre, size, colour, vel, axis, rate)."""
    rng = np.random.default_rng(seed)
    u, v, n = table_frame()
    colours = [(220, 40, 40), (40, 200, 60), (50, 80, 230), (230, 200, 30), (200, 40, 200), (30, 200, 210), (240, 130, 20), (130, 60, 220)]
    objs = []
    cols = int(np.ceil(np.sqrt(k)))
    for i in range(k):
        a = (i % cols - (cols - 1) / 2.0) * (0.9 / max(cols, 1)) if k > 1 else 0.0
        b = (i // cols - (cols - 1) / 2.0) * (0.55 / max(cols, 1)) if k > 1 else 0.0
        if k == 1:
            size = np.array([0.30, 0.24, 0.20])
        else:
            size = rng.uniform(0.08, 0.20, size=3) * (0.9 if k > 4 else 1.2)
        kind = "box" if (i % 3) != 2 else "sphere"
        h = size[2] / 2 if kind == "box" else size[0] / 2
        centre = _TABLE_P + a * u + b * v + (h + 0.002) * n
        # box axes: aligned with the table frame, yawed about the table normal
        R0 = np.stack([u, v, n], axis=1) @ _rot([0, 0, 1], rng.uniform(-0.6, 0.6))
        objs.append(dict(kind=kind, centre=centre, size=size, colour=colours[i % len(colours)], R0=R0,
                         vel=(0.02 * (u * np.cos(0.7 * i) + v * np.sin(0.7 * i))), axis=n, rate=np.deg2rad(2.0)))
    return objs


def object_pose(obj, frame, period=20):
    """Pose (R, c) at a frame: constant velocity 2 cm/frame and 2 deg/frame, reversing every `period`
    frames so that long runs stay on the table."""
    ph = frame % (2 * period)
    s = ph if ph <= period else 2 * period - ph
    c = obj["centre"] + s * obj["vel"]
    R = _rot(obj["axis"], s * obj["rate"]) @ obj["R0"]
    return R, c


def render(frame=0, objects=None, sensor=KINECT2_SD, seed=0xC0FFEE, noise=True, holes=0.05, camera=None):
    """Returns (points[H*W] POINT, obj_id[H*W] int8 (-1 = background/none)).

    The scene (table, wall, objects) is defined in the frame of the default camera.  `camera` = (R, t), the pose of
    another camera in that frame (world-from-camera: p_world = R p_cam + t), ray-casts the same scene from there; the
    points are then in that camera's optical frame."""
    if objects is None:
        objects = default_objects(1)
    W, H, f, cx, cy = sensor["width"], sensor["height"], sensor["f"], sensor["cx"], sensor["cy"]
    rng = np.random.default_rng(seed + 7919 * frame)
    uu, vv = np.meshgrid(np.arange(W, dtype=np.float64), np.arange(H, dtype=np.float64))
    d = np.stack([(uu - cx) / f, (vv - cy) / f, np.ones_like(uu)], axis=-1).reshape(-1, 3)
    d_cam = d
    # rays o + t d: t is the depth along the camera's optical axis (its z component of d is 1 in the camera frame)
    o = None
    if camera is not None:
        Rc, o = np.asarray(camera[0], dtype=np.float64), np.asarray(camera[1], dtype=np.float64)
        d = d_cam @ Rc.T
    n_px = d.shape[0]
    t_best = np.full(n_px, np.inf)
    colour = np.zeros((n_px, 3), dtype=np.float64)
    oid = np.full(n_px, -1, dtype=np.int8)

    def hit(t, col, ident, mask=None):
        m = (t > 0.05) & (t < t_best)
        if mask is not None:
            m &= mask
        t_best[m] = t[m]
        colour[m] = col
        oid[m] = ident

    # back wall z = 3.5
    if o is None:
        hit(np.full(n_px, 3.5), (200, 200, 190), -1)
    else:
        with np.errstate(divide="ignore", invalid="ignore"):
            tw = (3.5 - o[2]) / d[:, 2]
        hit(np.where(np.isfinite(tw), tw, -1.0), (200, 200, 190), -1)
    # table: bounded rectangle in the plane
    u, v, n = table_frame()
    denom = d @ n
    with np.errstate(divide="ignore", invalid="ignore"):
        t = ((_TABLE_P if o is None else _TABLE_P - o) @ n) / denom
    P = (d * t[:, None] if o is None else o + d * t[:, None]) - _TABLE_P
    inb = (np.abs(P @ u) < 0.85) & (np.abs(P @ v) < 0.60) & np.isfinite(t)
    hit(np.where(np.isfinite(t), t, -1.0), (120, 100, 80), -1, inb)
    for k, ob in enumerate(objects):
        R, c = object_pose(ob, frame)
        if o is not None:
            c = c - o  # the ray origin at 0
        if ob["kind"] == "sphere":
            r = ob["size"][0] / 2
            b = d @ c
            a = np.einsum("ij,ij->i", d, d)
            disc = b * b - a * (c @ c - r * r)
            with np.errstate(invalid="ignore"):
                t = (b - np.sqrt(disc)) / a
            hit(np.where(disc > 0, t, -1.0), ob["colour"], k)
        else:
            # ray (origin 0) in box frame: o = -R^T c, dir = R^T d ; slab test
            dl = d @ R
            ol = -(R.T @ c)
            half = ob["size"] / 2
            with np.errstate(divide="ignore", invalid="ignore"):
                t1 = (-half - ol) / dl
                t2 = (half - ol) / dl
            tn = np.max(np.minimum(t1, t2), axis=1)
            tf = np.min(np.maximum(t1, t2), axis=1)
            ok = (tn <= tf) & (tn > 0)
            # shade faces slightly differently so HSV coherence has something to see
            face = np.argmax(np.minimum(t1, t2), axis=1)
            col = np.asarray(ob["colour"], dtype=np.float64)[None, :] * (1.0 - 0.12 * face[:, None])
            m = ok & (tn < t_best)
            t_best[m] = tn[m]
            colour[m] = col[m]
            oid[m] = k
    z = t_best.copy()
    if noise:
        with np.errstate(invalid="ignore"):  # inf depth (rays of other viewpoints that hit nothing)
            z = z + rng.normal(0.0, 1.0, n_px) * 0.0015 * z * z
        colour = np.clip(colour + rng.uniform(-10, 10, colour.shape), 0, 255)
    pts = np.zeros(n_px, dtype=POINT)
    with np.errstate(invalid="ignore"):  # rays that hit nothing (other viewpoints): inf * 0, dropped below
        xyz = d_cam * z[:, None]
    bad = ~np.isfinite(z)
    if holes > 0:
        bad |= rng.random(n_px) < holes
    xyz[bad] = np.nan
    oid[bad] = -1
    pts["x"], pts["y"], pts["z"] = xyz[:, 0], xyz[:, 1], xyz[:, 2]
    c8 = colour.astype(np.uint32)
    pts["rgba"] = (255 << 24) | (c8[:, 0] << 16) | (c8[:, 1] << 8) | c8[:, 2]
    return pts, oid


def look_at(eye, target, up):
    """World-from-camera pose (R, t) of a camera at `eye` whose optical axis points at `target` (optical frame: x right,
    y down, z forward) with `up` up in its image."""
    eye, target, up = (np.asarray(a, dtype=np.float64) for a in (eye, target, up))
    z = target - eye
    z /= np.linalg.norm(z)
    x = np.cross(-up, z)
    x /= np.linalg.norm(x)
    y = np.cross(z, x)
    return np.stack([x, y, z], axis=1), eye


def side_camera():
    """A second viewpoint of the table: 1.3 m to its side along the table's u axis and 0.55 m above it, looking at its
    centre.  Returns the world-from-camera pose (R, t) that render(camera=...) takes."""
    u, v, n = table_frame()
    return look_at(_TABLE_P + 1.3 * u + 0.55 * n, _TABLE_P + 0.1 * n, n)


def pose_matrix(camera):
    """The 4x4 matrix of a world-from-camera pose (R, t): p_world = M @ [p_cam, 1]."""
    m = np.eye(4)
    m[:3, :3], m[:3, 3] = camera[0], camera[1]
    return m


def depth_images(pts, sensor=KINECT2_SD):
    """A rendered frame as the registered images kinect2_bridge publishes next to the points topic: returns
    (depth (H, W) uint16 millimetres, bgr (H, W, 3) uint8, K 3x3 float64 of camera_info).  z is rounded to the
    millimetre; a pixel without a reading (z NaN, or outside 1..65535 mm) is 0."""
    W, H, f, cx, cy = sensor["width"], sensor["height"], sensor["f"], sensor["cx"], sensor["cy"]
    with np.errstate(invalid="ignore"):
        mm = np.rint(np.asarray(pts["z"], dtype=np.float64) * 1000.0)
        ok = (mm >= 1) & (mm <= 65535)
    depth = np.where(ok, mm, 0).astype(np.uint16).reshape(H, W)
    rgba = np.asarray(pts["rgba"], dtype=np.uint32)
    bgr = np.stack([rgba & 0xff, (rgba >> 8) & 0xff, (rgba >> 16) & 0xff], axis=-1).astype(np.uint8).reshape(H, W, 3)
    K = np.array([[f, 0.0, cx], [0.0, f, cy], [0.0, 0.0, 1.0]])
    return depth, bgr, K


def model_points(pts, oid, k):
    """Raw model cloud of object k as create_model would return it (ref: src/create_model.cpp:209-230)."""
    m = (oid == k) & np.isfinite(pts["x"])
    return pts[m].copy()


def uniform_surface_scene(n_scene=100_000, n_model=5_000, seed=1):
    """Config C1: unorganised scene of n_scene points on a table plane + a box, and a model of n_model
    points sampled on the box (already centred on its centroid).  Returns (scene, model, centre)."""
    rng = np.random.default_rng(seed)
    u, v, n = table_frame()
    size = np.array([0.30, 0.24, 0.20])
    R = np.stack([u, v, n], axis=1)
    c = _TABLE_P + (size[2] / 2) * n

    def box_surface(m):
        areas = np.array([size[1] * size[2], size[0] * size[2], size[0] * size[1]])
        faces = rng.choice(3, size=m, p=areas / areas.sum())
        q = rng.uniform(-0.5, 0.5, size=(m, 3)) * size
        sign = np.where(rng.random(m) < 0.5, -0.5, 0.5)
        q[np.arange(m), faces] = sign * size[faces]
        return q

    n_box = n_scene // 5
    box = box_surface(n_box) @ R.T + c
    a = rng.uniform(-0.85, 0.85, n_scene - n_box)
    b = rng.uniform(-0.60, 0.60, n_scene - n_box)
    tab = _TABLE_P + a[:, None] * u + b[:, None] * v
    xyz = np.concatenate([box, tab]) + rng.normal(0, 0.001, (n_scene, 3))
    scene = np.zeros(n_scene, dtype=POINT)
    scene["x"], scene["y"], scene["z"] = xyz[:, 0], xyz[:, 1], xyz[:, 2]
    col = np.concatenate([np.tile([[220, 40, 40]], (n_box, 1)), np.tile([[120, 100, 80]], (n_scene - n_box, 1))])
    col = np.clip(col + rng.integers(-10, 11, col.shape), 0, 255).astype(np.uint32)
    scene["rgba"] = (255 << 24) | (col[:, 0] << 16) | (col[:, 1] << 8) | col[:, 2]
    perm = rng.permutation(n_scene)
    scene = scene[perm]
    mq = box_surface(n_model) @ R.T
    model = np.zeros(n_model, dtype=POINT)
    model["x"], model["y"], model["z"] = mq[:, 0], mq[:, 1], mq[:, 2]
    model["rgba"] = (255 << 24) | (220 << 16) | (40 << 8) | 40
    return scene, model, c.astype(np.float32)


def draws(slots, stride, seed=1234):
    """Injected RNG draw arrays shared by oracle and GPU (SURVEY A.9): selection uniforms [slots,stride],
    standard normals [slots,stride,6], motion uniforms [slots,stride]."""
    rng = np.random.default_rng(seed)
    usel = rng.random((slots, stride), dtype=np.float32)
    usel = np.minimum(usel, np.float32(1.0 - 2 ** -24))
    normals = rng.standard_normal((slots, stride, 6), dtype=np.float32)
    umot = rng.random((slots, stride), dtype=np.float32)
    return usel, normals, umot


def to_pcl32(pts):
    """16-byte packed points -> the 32-byte pcl::PointXYZRGBA layout (x,y,z,1.0f, rgba, pad[3])."""
    out = np.zeros(len(pts), dtype=np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("w", "<f4"), ("rgba", "<u4"), ("pad", "<u4", (3,))]))
    out["x"], out["y"], out["z"], out["w"], out["rgba"] = pts["x"], pts["y"], pts["z"], 1.0, pts["rgba"]
    return out
