"""The exact nearest-neighbour search on adversarial geometry, against the oracle's brute force.

The parity claim of the exact search is the brute-force answer bit for bit: same index, same squared distance, ties to
the lower input index (DESIGN §3, §5).  Random scenes about 1.2 m from the origin almost never reach the fp32 safety
rules that carry it, so every case here is built to reach one of them:

  lattice faces     points and queries exactly on fine-cell and octant faces (the rounding slack of the list build)
  equidistant       distinct points at bit-equal distance from a query, the lower index in another cell (tie order,
                    bisector tolerance, pairwise pruning)
  far scenes        coordinates at 8 m and 100 m, where an ulp is 8x and 64x larger (relative slacks and margins)
  max distance      points at exactly float(maximum_distance_^2) and one ulp either side (the distance cut lim2)
  crop faces        points just outside the crop box inside the dilated index, nearer than any cropped point, and
                    points exactly on the (inclusive) faces
  overflow          a query whose cell has more list candidates than an extended list holds (the warp brute force)
  depth images      the millimetre-quantised clouds of fromDepthImage / fromDepthImages, raw and downsampled

The builders and their preconditions are plain numpy and oracle code.  The tests without the gpu mark check on the CPU
that every case has the property it targets, so that none of them quietly turns into one more random scene; the gpu
tests compare every query of 8-16 recorded particles with the oracle (NN_EXACT_BRUTE), with the candidate lists off
and forced on."""
import functools

import numpy as np
import pytest

import oracle
from pcl_tracking_b200 import synth
from tests import util

f32 = np.float32
W_RTOL = 1e-5
LIST_MODES = [0, 2]  # exact-NN candidate lists: never / always
K_LIST_KX = 1024     # entries of an extended candidate list (kListKX): a cell with more candidates has no list
U10 = 2.0 ** -10     # a binary unit: sums and differences of multiples of it (|x| < 2^14 units) are exact in fp32


class Case:
    def __init__(self, scene, model, parts, max_dist=0.1, res=0.01, use_hsv=True, iters=2):
        self.scene, self.model, self.parts = scene, model, parts
        self.max_dist, self.res, self.use_hsv, self.iters = max_dist, res, use_hsv, iters


# ------------------------------------------------------------------ host arithmetic (the fp32 contract)
def xyz(pts):
    return np.stack([pts["x"], pts["y"], pts["z"]], axis=1).astype(f32)


def points(xyz_, rng):
    rgba = (255 << 24) | rng.integers(0, 1 << 24, len(xyz_)).astype(np.uint32)
    return oracle.make_points(np.asarray(xyz_, dtype=f32), rgba)


def host_queries(model, parts):
    """(N, M, 3): the model moved by each particle's matrix, ((m0 x + m1 y) + m2 z) + m3 with every operation rounded."""
    mats = np.stack([oracle.particle_to_matrix([p[k] for k in ("x", "y", "z", "roll", "pitch", "yaw")]) for p in parts])
    x, y, z = model["x"].astype(f32), model["y"].astype(f32), model["z"].astype(f32)
    out = np.empty((len(parts), len(model), 3), dtype=f32)
    for r in range(3):
        m = mats[:, r, :, None]
        out[:, :, r] = ((m[:, 0] * x + m[:, 1] * y) + m[:, 2] * z) + m[:, 3]
    return out


def host_d2(q, p):
    d = (q - p).astype(f32)
    return (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]


def host_nn(q, p):
    """Brute force: (index of the first minimum = the lower index on ties, d2, number of distinct points at that d2)."""
    q = q.reshape(-1, 3)
    idx, best, ties = np.empty(len(q), np.int64), np.empty(len(q), f32), np.empty(len(q), np.int64)
    for a in range(0, len(q), 512):
        d2 = host_d2(q[a:a + 512, None, :], p[None, :, :])
        idx[a:a + 512] = np.argmin(d2, axis=1)
        best[a:a + 512] = d2.min(axis=1)
        for r, (row, b) in enumerate(zip(d2, best[a:a + 512])):
            ties[a + r] = len(np.unique(p[row == b], axis=0))
    return idx, best, ties


def lattice_float(k, inv2):
    """Per integer k, an fp32 x near k / inv2 with x * inv2 == k exactly: x lies on an octant face of the lattice."""
    x = (np.asarray(k, np.float64) / np.float64(inv2)).astype(f32)
    out = np.full(x.shape, np.nan, dtype=f32)
    for s in (0, 1, -1, 2, -2, 3, -3, 4, -4):
        y = x.copy()
        for _ in range(abs(s)):
            y = np.nextafter(y, f32(np.inf) if s > 0 else f32(-np.inf))
        hit = np.isnan(out) & ((y * inv2).astype(f32) == np.asarray(k, dtype=f32))
        out[hit] = y[hit]
    return out


def inv_leaf(res):
    return f32(1.0) / f32(res)  # as the index build computes it


def on_octant_face(v, res):
    inv2 = inv_leaf(res) * f32(2.0)
    s = (v.astype(f32) * inv2).astype(f32)
    return s == np.floor(s)


def oracle_weight(c):
    """The oracle's weight() of a case, nearest neighbours kept."""
    o = oracle.Tracker(kld=False)
    oracle.configure_like_reference(o, particle_num=len(c.parts), max_particle_num=len(c.parts), use_hsv=c.use_hsv, iteration_num=c.iters)
    o.set_d(oracle.MAX_DIST, c.max_dist)
    o.set_d(oracle.GRID_CELL, c.res)
    o.set_reference(c.model)
    o.set_input(c.scene)
    o.set_particles(c.parts)
    o.weight(keep_nn=True)
    return o


@functools.lru_cache(maxsize=None)
def run_oracle(key):
    """(case, oracle) of CASES[key[0]](*key[1:])."""
    c = CASES[key[0]](*key[1:])
    return c, oracle_weight(c)


def oracle_nn(c, o):
    """(N, M) scene indices and d2 of the oracle's nearest cropped neighbours (-1 / d2 kept where the crop is empty)."""
    cidx, _ = o.cropped()
    n, m = len(c.parts), len(c.model)
    idx, d2 = np.empty((n, m), np.int64), np.empty((n, m), f32)
    for p in range(n):
        oi, od = o.nn(p, m)
        idx[p] = np.where(oi >= 0, cidx[np.maximum(oi, 0)], -1)
        d2[p] = od
    return idx, d2


# ------------------------------------------------------------------ case 1: points and queries on lattice faces
def lattice_case(res, seed=0):
    rng = np.random.default_rng(seed)
    inv2 = inv_leaf(res) * f32(2.0)
    centre, half = np.array([0.11, -0.07, 1.23]), 0.06
    k0, k1 = np.floor((centre - half) * float(inv2)).astype(int), np.ceil((centre + half) * float(inv2)).astype(int)
    axes = [lattice_float(np.arange(k0[d], k1[d] + 1), inv2) for d in range(3)]
    axes = [a[np.isfinite(a)] for a in axes]  # (a few k have no such float: left out)
    assert all(len(a) > 0.5 * (k1[d] - k0[d] + 1) for d, a in enumerate(axes))

    def pick(n):
        return np.stack([axes[d][rng.integers(0, len(axes[d]), n)] for d in range(3)], axis=1)

    sc = np.unique(pick(3000), axis=0)
    # copies one ulp off the face along one axis, on either side
    cp = sc[rng.choice(len(sc), 600, replace=False)].copy()
    ax, up = rng.integers(0, 3, len(cp)), rng.random(len(cp)) < 0.5
    cp[np.arange(len(cp)), ax] = np.nextafter(cp[np.arange(len(cp)), ax], np.where(up, f32(np.inf), f32(-np.inf)).astype(f32))
    all_pts = np.concatenate([sc, cp])
    scene = points(all_pts[rng.permutation(len(all_pts))], rng)
    model = points(pick(220), rng)
    # particles: the model as it is (the queries are the lattice points), moved by lattice steps (exact sums of face
    # floats), and turned by small angles
    steps = [lattice_float(np.array([k]), inv2)[0] for k in (-2, -1, 1, 2)]
    assert np.isfinite(steps).all()
    states = [[0, 0, 0, 0, 0, 0]]
    for k in range(7):
        states.append([steps[k % 4] * (d == k % 3) for d in range(3)] + [0, 0, 0])
    for k in range(4):
        states.append([0, 0, 0] + list(rng.normal(0, 0.01, 3)))
    return Case(scene, model, oracle.make_particles(np.array(states, dtype=f32), np.full(len(states), 1.0 / len(states), dtype=f32)), res=res)


# ------------------------------------------------------------------ case 2: distinct points at bit-equal distances
def _norm25():
    v = [(a, b, c) for a in range(-5, 6) for b in range(-5, 6) for c in range(-5, 6) if a * a + b * b + c * c == 25]
    return np.array(v, dtype=np.float64)


def equidistant_case(seed=0):
    """Queries and points on the 2^-10 m lattice (every sum and difference exact): around each query of the unmoved
    particle, 2-4 points at the same integer offset norm (|v| = 5 units, d2 bit-equal); the lower-index ones lie in
    other fine cells than the query, the last one in the query's own cell."""
    rng = np.random.default_rng(seed)
    res, s = 0.01, 32  # fine cell 1 cm; grid spacing 32 units = 3.125 cm
    inv = float(inv_leaf(res))
    base = np.round((np.floor(np.array([0.11, -0.07, 1.23]) * 100) + np.array([0.25, 0.30, 0.70])) * 0.01 / U10)
    g = np.stack(np.meshgrid(*[np.arange(4)] * 3, indexing="ij"), -1).reshape(-1, 3)
    model_u = base + s * g
    model = points(model_u * U10, rng)
    q = xyz(model)
    vs = _norm25()
    cell = lambda p: np.floor((p.astype(f32) * f32(inv)).astype(f32))
    twins_lo, twins_hi = [], []
    for qu, qf in zip(model_u, q):
        p = ((qu + vs) * U10).astype(f32)
        own = np.all(cell(p) == cell(qf[None]), axis=1)
        lo = rng.permutation(np.flatnonzero(~own))[:rng.integers(1, 4)]
        hi = rng.permutation(np.flatnonzero(own))[:1]
        twins_lo.append(p[lo])
        twins_hi.append(p[hi])
    # clutter of the crop box, at least 1.2 cm from every lattice point the exact particles move a query to
    lo_box, hi_box = (base - 2 * s) * U10, (base + 5 * s) * U10
    cl = rng.uniform(lo_box, hi_box, (6000, 3))
    lat = (base + s * np.stack(np.meshgrid(*[np.arange(-1, 5)] * 3, indexing="ij"), -1).reshape(-1, 3)) * U10
    far = np.array([np.min(np.linalg.norm(lat - c, axis=1)) for c in cl]) > 0.012
    cl = cl[far][:1500].astype(f32)
    # lower-index twins first, then clutter, then the own-cell twins
    scene = points(np.concatenate(twins_lo + [cl] + twins_hi), rng)
    shifts = [(0, 0, 0), (s, 0, 0), (0, s, 0), (0, 0, s), (-s, 0, 0), (s, s, 0), (0, -s, s), (s, 0, -s)]
    states = [[0.0, 0.0, 0.0] + [0.0] * 3 for _ in shifts]
    for st, sh in zip(states, shifts):
        st[:3] = list(np.array(sh) * U10)
    for _ in range(4):
        states.append(list(rng.normal(0, 0.003, 3)) + list(rng.normal(0, 0.02, 3)))
    return Case(scene, model, oracle.make_particles(np.array(states, dtype=f32), np.full(len(states), 1.0 / len(states), dtype=f32)), res=res)


# ------------------------------------------------------------------ case 3: far scenes
FAR_OFFSETS = {"kinect_right": (3.0, 0.2, 7.0), "kinect_left": (-3.0, -0.2, 7.0), "world_100m": (100.0, 100.0, 100.0)}


def far_case(where, seed=4):
    off = np.array(FAR_OFFSETS[where], dtype=f32)
    scene, model, centre = util.small_case(seed, n_scene=3000, n_model=200)
    for d, k in enumerate("xyz"):
        scene[k] = (scene[k] + off[d]).astype(f32)
    parts = util.particles_around(centre + off, 12, seed=seed + 100)
    return Case(scene, model, parts)


# ------------------------------------------------------------------ case 4: the maximum-distance boundary
def boundary_targets(max_dist):
    """float(max_d2) (round to nearest) and its two fp32 neighbours, with whether each is a match ((double)d2 < max_d2)."""
    md2 = max_dist * max_dist
    t = f32(md2)
    ts = [t, np.nextafter(t, f32(np.inf)), np.nextafter(t, f32(0))]
    return [(x, float(x) < md2) for x in ts]


def point_at_d2(q, target, sx, sy):
    """An fp32 point p with host_d2(q, p) == target exactly: offset ~sqrt(target) along x (sign sx), 2 mm along y."""
    dy0 = 2e-3
    dx0 = np.sqrt(float(target) - dy0 * dy0)
    px0, py0 = f32(float(q[0]) - sx * dx0), f32(float(q[1]) - sy * dy0)
    px = (np.float64(px0) + np.arange(-40, 41) * np.float64(np.spacing(px0))).astype(f32)
    py = (np.float64(py0) + np.arange(-400, 401) * np.float64(np.spacing(py0))).astype(f32)
    P = np.stack(np.broadcast_arrays(px[:, None], py[None, :], np.full((1, 1), q[2], dtype=f32)), -1).reshape(-1, 3)
    hit = np.flatnonzero(host_d2(q[None, :], P) == target)
    assert len(hit), (q, target)
    return P[hit[len(hit) // 2]]


def boundary_case(max_dist, seed=0):
    """Queries on a grid 0.375 m apart (exact binary coordinates); at each, ONE scene point at d2 = float(max_d2) or one
    ulp either side (cycled over the grid); clutter at least 0.2 m from every query."""
    rng = np.random.default_rng(seed)
    s = 0.375
    g = np.stack(np.meshgrid(np.arange(3), np.arange(3), np.arange(2), indexing="ij"), -1).reshape(-1, 3)
    model = points((g - g.mean(0)) * s, rng)
    c = np.array([112, -72, 1264]) * U10
    shifts = [(0, 0, 0), (1, 0, 0), (-1, 0, 0), (0, 1, 0), (0, -1, 0), (0, 0, 1), (1, 1, 0), (0, -1, 1)]
    states = [list(c + np.array(sh) * s) + [0.0] * 3 for sh in shifts]
    for _ in range(4):
        states.append(list(c + rng.normal(0, 0.002, 3)) + list(rng.normal(0, 0.01, 3)))
    parts = oracle.make_particles(np.array(states, dtype=f32), np.full(len(states), 1.0 / len(states), dtype=f32))
    locs = np.unique(host_queries(model, parts[:len(shifts)]).reshape(-1, 3), axis=0)
    targets = boundary_targets(max_dist)
    mid = locs.mean(0)
    pts = []
    for k, q in enumerate(locs):
        sx, sy = (1.0 if q[0] > mid[0] else -1.0), (1.0 if q[1] > mid[1] else -1.0)  # toward the middle: inside the crop
        pts.append(point_at_d2(q, targets[k % 3][0], sx, sy))
    lo, hi = locs.min(0), locs.max(0)
    cl = rng.uniform(lo, hi, (3000, 3)).astype(f32)
    cl = cl[np.array([np.min(np.linalg.norm(locs - p, axis=1)) for p in cl]) > 0.2][:600]
    allp = np.concatenate([np.array(pts, dtype=f32), cl])
    scene = points(allp[rng.permutation(len(allp))], rng)
    return Case(scene, model, parts, max_dist=max_dist, res=0.02)


# ------------------------------------------------------------------ case 5: crop faces, and a cell without a list
def crop_faces_case(seed=8):
    """A small_case scene; next to every query within 4 mm of a face of the crop box, a point just beyond that face
    (inside the 3 cm the index is dilated by when a compute() has two iterations) and nearer than any cropped point,
    and a point exactly on the face."""
    rng = np.random.default_rng(seed)
    scene, model, centre = util.small_case(seed, n_scene=3000, n_model=200)
    parts = util.particles_around(centre, 12, seed=seed + 100)
    q = host_queries(model, parts).reshape(-1, 3)
    box = np.concatenate([q.min(0), q.max(0)])
    extra = []
    for d in range(3):
        for side, face in ((-1.0, box[d]), (1.0, box[3 + d])):
            near = q[np.abs(q[:, d] - face) <= 0.004]
            for p in near:
                out = p.copy()
                out[d] = f32(face + side * rng.uniform(5e-5, 3e-4))  # just beyond the face
                extra.append(out)
                on = p.copy()
                on[(d + 1) % 3] = f32(on[(d + 1) % 3] + rng.uniform(-0.004, 0.004))
                on[d] = face  # exactly on the face: cropped (the limits are inclusive)
                extra.append(on)
            far = p.copy()
            far[d] = np.nextafter(f32(face), f32(side * np.inf))  # one ulp beyond the face
            extra.append(far)
    extra = points(np.array(extra, dtype=f32), rng)
    allp = np.concatenate([scene, extra])
    return Case(allp[rng.permutation(len(allp))], model, parts)


def overflow_case(seed=9, n_shell=1500, radius=0.04):
    """A small_case scene plus a model point at the model origin (its query is the particle's translation, exactly) and
    a shell of n_shell > kListKX points at `radius` around particle 0's translation: the cell of that query has more
    list candidates than an extended list holds, so it has no list and the query is answered by brute force."""
    rng = np.random.default_rng(seed)
    scene, model, centre = util.small_case(seed, n_scene=3000, n_model=200)
    model = np.concatenate([model, points(np.zeros((1, 3)), rng)])
    parts = util.particles_around(centre, 12, seed=seed + 100, sigma_t=0.004)
    c0 = np.array([parts[0]["x"], parts[0]["y"], parts[0]["z"]], dtype=np.float64)
    v = rng.normal(size=(n_shell, 3))
    shell = points(c0 + radius * v / np.linalg.norm(v, axis=1, keepdims=True), rng)
    allp = np.concatenate([scene, shell])
    return Case(allp[rng.permutation(len(allp))], model, parts)


# ------------------------------------------------------------------ case 6: depth-image scenes
def _depth_model(cloud, oid, seed):
    rng = np.random.default_rng(seed)
    raw = synth.model_points(cloud, oid, 0)
    c = xyz(raw).astype(np.float64).mean(0).astype(f32)
    model = raw[rng.choice(len(raw), min(300, len(raw)), replace=False)].copy()
    for d, k in enumerate("xyz"):
        model[k] = (model[k] - c[d]).astype(f32)
    return model, c


@functools.lru_cache(maxsize=None)
def depth_frames(kind):
    """(camera dicts for fromDepthImages, host restatement of the organised / fused cloud, model, centre)."""
    from tests.test_gpu_depth import restate
    from tests.test_gpu_depth_cameras import restate_fused
    s = synth.KINECT2_SD
    objs = synth.default_objects(1)
    pts, oid = synth.render(0, objs, sensor=s)
    d0, c0, K0 = synth.depth_images(pts, s)
    cam0 = dict(depth=d0, bgr=c0, fx=K0[0, 0], fy=K0[1, 1], cx=K0[0, 2], cy=K0[1, 2], pose=None)
    model, centre = _depth_model(restate(d0, c0, cam0["fx"], cam0["fy"], cam0["cx"], cam0["cy"]), oid, 3)
    if kind == "one_camera":
        cams = [cam0]
        cloud = restate(d0, c0, cam0["fx"], cam0["fy"], cam0["cx"], cam0["cy"])
    else:
        side = synth.side_camera()
        d1, c1, K1 = synth.depth_images(synth.render(0, objs, sensor=s, camera=side)[0], s)
        pose = synth.pose_matrix(side).astype(f32)
        cams = [cam0, dict(depth=d1, bgr=c1, fx=K1[0, 0], fy=K1[1, 1], cx=K1[0, 2], cy=K1[1, 2], pose=pose)]
        cloud = restate_fused(cams)
    return cams, cloud, model, centre


def depth_case(kind, seed=11):
    _, cloud, model, centre = depth_frames(kind)
    return Case(cloud, model, util.particles_around(centre, 12, seed=seed))


CASES = {"lattice": lattice_case, "equidistant": equidistant_case, "far": far_case, "boundary": boundary_case,
         "crop_faces": crop_faces_case, "overflow": overflow_case, "depth": depth_case}
LATTICE_RES = [0.005, 0.01, 0.02]
BOUNDARY_DIST = [0.1, 0.125]


# ------------------------------------------------------------------ preconditions (CPU: the oracle alone)
@pytest.mark.parametrize("res", LATTICE_RES)
def test_lattice_case_sits_on_octant_faces(res):
    c, o = run_oracle(("lattice", res))
    q = host_queries(c.model, c.parts).reshape(-1, 3)
    qf = on_octant_face(q, res)
    sf = on_octant_face(xyz(c.scene), res)
    assert qf.all(axis=1).mean() >= 0.35  # the unmoved and the lattice-stepped particles: all three coordinates
    assert qf.any(axis=1).mean() >= 0.6
    assert sf.all(axis=1).mean() >= 0.6 and (sf.sum(axis=1) == 2).sum() >= 400  # + the one-ulp copies
    idx, d2 = oracle_nn(c, o)
    assert (d2.astype(np.float64) < c.max_dist ** 2).mean() > 0.9


def test_equidistant_case_has_bit_equal_twins():
    c, o = run_oracle(("equidistant",))
    q = host_queries(c.model, c.parts)
    cidx, cpts = o.cropped()
    idx, d2 = oracle_nn(c, o)
    hidx, hd2, ties = host_nn(q.reshape(-1, 3), xyz(cpts))
    np.testing.assert_array_equal(cidx[hidx], idx.ravel())  # the host brute force is the oracle's
    np.testing.assert_array_equal(hd2, d2.ravel())
    assert (ties >= 2).sum() >= 150
    # particle 0: every query has 2-4 distinct points at the same d2; the winner (lower index) lies in another fine cell
    inv = inv_leaf(c.res)
    t0 = ties[:len(c.model)]
    assert np.all((t0 >= 2) & (t0 <= 4))
    win = xyz(c.scene)[idx[0]]
    assert np.all(np.any(np.floor(win * inv) != np.floor(q[0] * inv), axis=1))
    # ... and the last of the tied points lies in the query's own cell
    sc = xyz(c.scene)
    for j in range(len(c.model)):
        dd = host_d2(q[0, j][None], sc)
        last = np.flatnonzero(dd == d2[0, j])[-1]
        assert np.all(np.floor(sc[last] * inv) == np.floor(q[0, j] * inv))


@pytest.mark.parametrize("where", list(FAR_OFFSETS))
def test_far_case_is_far(where):
    c, o = run_oracle(("far", where))
    q = host_queries(c.model, c.parts).reshape(-1, 3)
    assert np.all(np.abs(q).max(axis=1) >= 8.0)  # an ulp of a coordinate is at least 8x the ulp at 1.2 m
    assert np.all(np.spacing(np.abs(q).max(axis=1)) >= 8 * np.spacing(f32(1.2)))
    idx, d2 = oracle_nn(c, o)
    assert (d2.astype(np.float64) < c.max_dist ** 2).mean() > 0.5


@pytest.mark.parametrize("max_dist", BOUNDARY_DIST)
def test_boundary_case_sits_on_the_cut(max_dist):
    c, o = run_oracle(("boundary", max_dist))
    targets = boundary_targets(max_dist)
    # the cut: the round-to-nearest float of max_d2 counts for 0.1 (it lies below 0.1^2) and not for 0.125 (it is
    # 0.125^2 exactly); the float above it never counts, the float below it always does
    assert [m for _, m in targets] == ([True, False, True] if max_dist == 0.1 else [False, False, True])
    idx, d2 = oracle_nn(c, o)
    exact = d2[:8].ravel()  # the particles moved by whole grid steps
    for t, _ in targets:
        assert (exact == t).sum() >= 20
    assert np.isin(exact, [t for t, _ in targets]).mean() > 0.95


def test_crop_faces_case_has_nearer_points_outside_the_crop():
    c, o = run_oracle(("crop_faces",))
    box = o.aabb()
    q = host_queries(c.model, c.parts).reshape(-1, 3)
    np.testing.assert_array_equal(np.concatenate([q.min(0), q.max(0)]), box)
    idx, d2 = oracle_nn(c, o)
    sc = xyz(c.scene)
    inside = np.all((sc >= box[:3]) & (sc <= box[3:]), axis=1)
    dil = np.all((sc >= box[:3] - 0.03) & (sc <= box[3:] + 0.03), axis=1)
    assert (np.any(sc == box[:3], axis=1) | np.any(sc == box[3:], axis=1)).sum() >= 20  # points exactly on the faces
    # the full scene's nearest point is outside the crop box (within the dilation) and nearer than the cropped one
    fidx, fd2, _ = host_nn(q, sc)
    out = ~inside[fidx] & dil[fidx] & (fd2 < d2.ravel())
    assert out.sum() >= 30
    assert np.all(inside[idx.ravel()])


def test_overflow_case_has_a_crowded_cell():
    c, o = run_oracle(("overflow",))
    q0 = host_queries(c.model, c.parts)[0, -1]
    assert np.array_equal(q0, np.array([c.parts[0][k] for k in "xyz"], dtype=f32))
    cidx, cpts = o.cropped()
    d = np.sqrt(host_d2(q0[None], xyz(cpts)).astype(np.float64))
    assert (np.abs(d - 0.04) < 1e-4).sum() > K_LIST_KX + 200  # the whole shell is cropped
    assert (d < 0.04 - 1e-4).sum() == 0
    idx, d2 = oracle_nn(c, o)
    assert abs(np.sqrt(float(d2[0, -1])) - 0.04) < 1e-4


@pytest.mark.parametrize("kind", ["one_camera", "two_cameras"])
def test_depth_case_is_quantised(kind):
    c, o = run_oracle(("depth", kind))
    n0 = synth.KINECT2_SD["width"] * synth.KINECT2_SD["height"]
    # camera 0 (the common frame): organised, holes as NaN, depth in whole millimetres -- every z is float(k) * 0.001f
    cam0 = c.scene[:n0]
    sc = cam0[np.isfinite(cam0["z"])]
    assert len(c.scene) == (1 if kind == "one_camera" else 2) * n0 and len(sc) < n0
    k = np.round(sc["z"].astype(np.float64) * 1000)
    assert np.array_equal(sc["z"], (k.astype(f32) * f32(0.001)).astype(f32))
    assert len(np.unique(sc["z"])) < 0.02 * len(sc)
    idx, d2 = oracle_nn(c, o)
    assert (d2.astype(np.float64) < c.max_dist ** 2).mean() > 0.5


# ------------------------------------------------------------------ GPU comparisons
def _compare(c, o, lists, cloud=None):
    from pcl_tracking_b200 import pcl
    g, _ = util.make_pair(kld=False, particle_num=len(c.parts), use_hsv=c.use_hsv, max_dist=c.max_dist, search_res=c.res, iteration_num=c.iters)
    g.setReferenceCloud(c.model)
    g.setInputCloud(cloud if cloud is not None else pcl.PointCloud(c.scene))
    g.setParticles(c.parts)
    g.setDebugNN(len(c.parts))
    g.setCandidateLists(lists)
    g.weight()
    if lists == 2:
        assert g.indexInfo()["use_lists"] == 1
    np.testing.assert_array_equal(g.aabb(), o.aabb())
    cidx, _ = o.cropped()
    assert g.croppedCount() == len(cidx)
    want_i, want_d = oracle_nn(c, o)
    matched = (want_i >= 0) & (want_d.astype(np.float64) < c.max_dist * c.max_dist)  # what the coherence counts
    m = len(c.model)
    for p in range(len(c.parts)):
        gi, gd = g.nn(p, m)
        wi = np.where(matched[p], want_i[p], -1)
        bad = np.flatnonzero(gi != wi)
        assert len(bad) == 0, ("particle", p, "queries", bad[:8], "gpu", gi[bad[:8]], "oracle", wi[bad[:8]], want_d[p, bad[:8]])
        np.testing.assert_array_equal(gd[matched[p]], want_d[p][matched[p]])
    assert matched.any()
    np.testing.assert_allclose(g.rawWeights(), o.raw_weights(), rtol=W_RTOL, atol=0)


@pytest.mark.gpu
@pytest.mark.parametrize("lists", LIST_MODES)
@pytest.mark.parametrize("res", LATTICE_RES)
def test_gpu_lattice_faces(res, lists):
    _compare(*run_oracle(("lattice", res)), lists)


@pytest.mark.gpu
@pytest.mark.parametrize("lists", LIST_MODES)
def test_gpu_equidistant_twins(lists):
    _compare(*run_oracle(("equidistant",)), lists)


@pytest.mark.gpu
@pytest.mark.parametrize("lists", LIST_MODES)
@pytest.mark.parametrize("where", list(FAR_OFFSETS))
def test_gpu_far_scenes(where, lists):
    _compare(*run_oracle(("far", where)), lists)


@pytest.mark.gpu
@pytest.mark.parametrize("lists", LIST_MODES)
@pytest.mark.parametrize("max_dist", BOUNDARY_DIST)
def test_gpu_max_distance_boundary(max_dist, lists):
    _compare(*run_oracle(("boundary", max_dist)), lists)


@pytest.mark.gpu
@pytest.mark.parametrize("lists", LIST_MODES)
def test_gpu_crop_faces(lists):
    _compare(*run_oracle(("crop_faces",)), lists)


@pytest.mark.gpu
@pytest.mark.parametrize("lists", LIST_MODES)
def test_gpu_cell_without_list(lists):
    _compare(*run_oracle(("overflow",)), lists)


@pytest.mark.gpu
@pytest.mark.parametrize("lists", LIST_MODES)
@pytest.mark.parametrize("kind", ["one_camera", "two_cameras"])
def test_gpu_depth_image_scene(kind, lists):
    """The device cloud of the depth ingest equals the host restatement bit for bit; tracking reads it organised (NaN
    holes included), then after PassThrough + the 1 cm voxel grid (the downloaded cloud is the oracle's input)."""
    from pcl_tracking_b200 import pcl
    cams, host, _, _ = depth_frames(kind)
    c, o = run_oracle(("depth", kind))
    cloud = pcl.PointCloud()
    if kind == "one_camera":
        cam = cams[0]
        cloud.fromDepthImage(cam["depth"], cam["bgr"], cam["fx"], cam["fy"], cam["cx"], cam["cy"])
    else:
        cloud.fromDepthImages(cams)
    assert np.array_equal(cloud.to_numpy().view(np.uint32), host.view(np.uint32))
    _compare(c, o, lists, cloud)
    vg = pcl.ApproximateVoxelGrid()
    vg.setLeafSize(0.01, 0.01, 0.01)
    vg.setPassThrough("z", 0.0, 10.0)
    vg.setInputCloud(cloud)
    ds = vg.filter()
    down = Case(ds.to_numpy(), c.model, c.parts)
    assert len(down.scene) > 1000
    _compare(down, oracle_weight(down), lists, ds)
