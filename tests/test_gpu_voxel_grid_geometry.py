"""The voxel-grid downsample (K1: PassThrough + voxel grid) on adversarial lattices, against an exact reference.

K1's claim is bit-exactness (DESIGN §0 a1-a2, §3): the voxels of the lattice floor(fp32(v) * fp32(1/leaf)), saturated
to the int32 range, in order of first appearance, each with its exact centroid rounded to fp32 and upstream's truncated
colour means.  Random clouds near the sensor reach few of the rules that carry that claim, so every case here is built
to reach one of them:

  lattice faces   points at k * leaf in fp32 and 1-2 ulp either side, where the fp32 product and exact division
                  disagree (six leaf sizes)
  signs and zero  +-0, denormals, +-1e-30 and -leaf * (1 - ulp): voxels 0 and -1 of every axis
  far keys        indices at +-2^20 (+-1), voxels 2^21 * k cells apart on one axis (one key each, not one per residue)
                  and products past +-2^31 (saturated), up to +-3.4e38
  hash            every point its own voxel, one voxel of 300 000 points (colour sums past 2^24), 300 voxels homed on
                  one slot near the end of the table (a probe chain that wraps), capacities either side of a table step
  order and tiles first points and rejected points on the 4096-point tile edges, n = k * 4096 +- 1, more than 1024
                  tiles (the second pass of the tile scan), eight fused qhd cameras
  limits          every field, lo == hi, lo > hi, infinite and NaN limits, NaN in the filtered field and in another
                  one; the same through pft_passthrough; removeZeroPoints / prepare_model at |c| = 0.01f
  graph cache     one (in, out) pair with leaf, limits and field changed between calls, double-buffered asynchronous
                  frames of different sizes, more (in, out) pairs than the cache holds

The reference (`reference`) is a numpy restatement written apart from the C++ oracle.  Its centroid is the exact sum
(math.fsum where fp64 additions could round) over the count; a CPU test checks that every voxel of every case sums
exactly in fp64 in any order, so the order in which the GPU's atomics land cannot matter, and pins the oracle to the
reference.  The other tests without the gpu mark check that each case has the property it was built for; the gpu tests
compare count, order, xyz bits and rgba bits."""
import functools
import math

import numpy as np
import pytest

import oracle
from pcl_tracking_b200 import pcl

f32 = np.float32
I32_MIN, I32_MAX = -2 ** 31, 2 ** 31 - 1
TILE = 4096                 # points per block of the ranking kernels (kTile)
F32_MAX = float(np.finfo(f32).max)


class Case:
    def __init__(self, pts, leaf=0.01, field=-1, lo=0.0, hi=0.0):
        self.pts, self.leaf, self.field, self.lo, self.hi = pts, leaf, field, lo, hi


# ------------------------------------------------------------------ the reference
def xyz(pts):
    return np.stack([pts["x"], pts["y"], pts["z"]], axis=1).astype(f32)


def points(xyz_, rng):
    return oracle.make_points(np.asarray(xyz_, dtype=f32), rng.integers(0, 1 << 32, len(xyz_), dtype=np.uint64).astype(np.uint32))


def inv_leaf(leaf):
    return f32(1.0) / f32(leaf)


def voxel_index(v, leaf):
    """floor(fp32(v) * fp32(1/leaf)), the product rounded to fp32, saturated to the int32 range (as int64)."""
    with np.errstate(over="ignore", invalid="ignore"):
        p = np.floor(np.asarray(v, dtype=f32) * inv_leaf(leaf))
    return np.clip(np.nan_to_num(p.astype(np.float64)), I32_MIN, I32_MAX).astype(np.int64)


def passes(pts, field, lo, hi):
    """Finite points, and !(v < lo || v > hi) on the filtered field (limits rounded to fp32, as the C ABI takes them)."""
    p = xyz(pts)
    ok = np.isfinite(p).all(axis=1)
    if field >= 0:
        with np.errstate(invalid="ignore"):
            v = p[:, field]
            ok &= ~((v < f32(lo)) | (v > f32(hi)))
    return ok


def voxel_ids(keys):
    """Rank of each row's voxel in order of first appearance, and the index of each voxel's first row."""
    if len(keys) == 0:
        return np.zeros(0, np.int64), np.zeros(0, np.int64)
    ids = np.zeros(len(keys), np.int64)
    for d in range(3):  # dense ids of (x), (x, y), (x, y, z): no product overflows
        _, col = np.unique(keys[:, d], return_inverse=True)
        _, ids = np.unique(ids * (col.max() + 1) + col, return_inverse=True)
    nv = ids.max() + 1
    first = np.full(nv, len(keys), np.int64)
    np.minimum.at(first, ids, np.arange(len(keys)))
    order = np.argsort(first)
    rank = np.empty(nv, np.int64)
    rank[order] = np.arange(nv)
    return rank[ids], first[order]


def voxel_sums(v, ids, nv):
    """(sums, order_free): per voxel the exact sum of the fp32 values `v` (the fp64 nearest to it), and whether fp64
    additions in every order give it: at most two terms, or the sum of |v| below 2^53 times the voxel's smallest ulp
    (every partial sum is then a multiple of that ulp that fp64 holds exactly)."""
    v64 = v.astype(np.float64)
    sums = np.bincount(ids, weights=v64, minlength=nv)  # in input order, from +0
    cnt = np.bincount(ids, minlength=nv)
    absum = np.bincount(ids, weights=np.abs(v64), minlength=nv)
    with np.errstate(over="ignore"):
        sp = np.spacing(np.abs(v)).astype(np.float64)  # inf at FLT_MAX, whose ulp is 2^104
    ulp = np.where(v64 != 0, np.minimum(sp, 2.0 ** 104), np.inf)
    umin = np.full(nv, np.inf)
    np.minimum.at(umin, ids, ulp)
    free = (cnt <= 2) | (absum * (1 + 2.0 ** -40) < 2.0 ** 53 * umin)
    for k in np.flatnonzero(~free):
        sums[k] = math.fsum(v64[ids == k]) + 0.0
    return sums, free


def reference(pts, leaf, field=-1, lo=0.0, hi=0.0, with_free=False):
    """The downsample K1 specifies, restated: (points, and per voxel whether its sums are order free)."""
    sel = pts[passes(pts, field, lo, hi)]
    p = xyz(sel)
    keys = np.stack([voxel_index(p[:, d], leaf) for d in range(3)], axis=1)
    ids, _ = voxel_ids(keys)
    nv = int(ids.max()) + 1 if len(ids) else 0
    cnt = np.bincount(ids, minlength=nv).astype(np.float64)
    out = np.zeros(nv, dtype=oracle.POINT)
    free = np.ones(nv, bool)
    for d, name in enumerate("xyz"):
        s, fr = voxel_sums(p[:, d], ids, nv)
        out[name] = (s / cnt).astype(f32)
        free &= fr
    rgba = sel["rgba"].astype(np.int64)
    fc = cnt.astype(f32)
    col = np.zeros(nv, np.uint32)
    for shift in (16, 8, 0):
        csum = np.bincount(ids, weights=(rgba >> shift) & 0xff, minlength=nv)
        col |= ((csum.astype(f32) / fc).astype(np.int64).astype(np.uint32)) << np.uint32(shift)
    out["rgba"] = col
    return (out, free) if with_free else out


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32).reshape(len(a), 4)


def assert_same(got, want):
    assert len(got) == len(want), "%d voxels, reference %d" % (len(got), len(want))
    bad = np.flatnonzero((bits(got) != bits(want)).any(axis=1))
    assert len(bad) == 0, "%d of %d voxels differ, first %s: got %s, reference %s" % (len(bad), len(want), bad[:4], got[bad[:3]], want[bad[:3]])


# ------------------------------------------------------------------ lattice helpers
def solve(idx, leaf, frac=0.5):
    """fp32 coordinates whose voxel index is `idx` (int array), started at (idx + frac) / inv and walked ulp by ulp."""
    idx = np.asarray(idx, np.int64)
    x = ((idx + frac) / np.float64(inv_leaf(leaf))).astype(f32)
    for _ in range(64):
        k = voxel_index(x, leaf)
        if np.array_equal(k, idx):
            break
        x = np.where(k < idx, np.nextafter(x, f32(np.inf)), np.where(k > idx, np.nextafter(x, f32(-np.inf)), x))
    return x


def ulps(x, s):
    x = np.asarray(x, f32)
    for _ in range(abs(s)):
        x = np.nextafter(x, f32(np.inf) if s > 0 else f32(-np.inf))
    return x


def table_size(cap):
    """Slots of the voxel hash for an input of capacity `cap` (run_voxel_grid)."""
    h = 1024
    while h < 2 * cap:
        h <<= 1
    return h


def voxel_hash(ix, iy, iz):
    """The voxel hash of k1_insert_kernel restated: (ix << 32 | iy) ^ iz * golden, then MurmurHash3's fmix64."""
    u = lambda a: (np.asarray(a, np.int64) & 0xffffffff).astype(np.uint64)
    with np.errstate(over="ignore"):
        k = (u(ix) << np.uint64(32)) | u(iy)
        k ^= u(iz) * np.uint64(0x9e3779b97f4a7c15)
        k ^= k >> np.uint64(33)
        k *= np.uint64(0xff51afd7ed558ccd)
        k ^= k >> np.uint64(33)
        k *= np.uint64(0xc4ceb9fe1a85ec53)
        k ^= k >> np.uint64(33)
    return k & np.uint64(0xffffffff)


def in_voxels(idx, leaf, rng):
    """One fp32 point inside each voxel of the (n, 3) index array, at a random place well inside it."""
    return np.stack([solve(idx[:, d], leaf, rng.uniform(0.1, 0.9, len(idx))) for d in range(3)], axis=1)


# ------------------------------------------------------------------ cases
LATTICE_LEAVES = [0.01, 0.005, 0.003, 0.0025, 1e-4, 0.1]


@functools.lru_cache(maxsize=None)
def lattice(leaf):
    """k * leaf in fp32 for k in [-3000, 3000) and 1-2 ulp either side, on every axis; the five variants of one k share
    their y and z, so the voxels on a face hold points from both sides of it."""
    rng = np.random.default_rng(int(leaf * 1e5))
    k = np.arange(-3000, 3000)
    base = k.astype(f32) * f32(leaf)
    vals = np.stack([ulps(base, s) for s in (0, 1, -1, 2, -2)], axis=1)  # (6000, 5)
    kx = np.repeat(np.arange(6000), 5)
    v = np.tile(np.arange(5), 6000)
    p = np.stack([vals[kx, v], vals[(kx * 7919) % 6000, (kx // 5) % 5], vals[(kx * 104729) % 6000, (kx // 25) % 5]], axis=1)
    return Case(points(p[rng.permutation(len(p))], rng), leaf, 2, -20.0, 20.0)


def signs_zero_values(leaf):
    tiny = [0.0, -0.0, 2.0 ** -149, -2.0 ** -149, 2.0 ** -140, -2.0 ** -140, 2.0 ** -126, -2.0 ** -126]
    small = [1e-30, -1e-30]
    l32 = f32(leaf)
    big = [float(np.nextafter(-l32, f32(0))), float(-l32), float(np.nextafter(l32, f32(0))), float(ulps(-l32, -1))]
    return [(v, 0) for v in tiny] + [(v, 1) for v in small] + [(v, 2) for v in big]


@functools.lru_cache(maxsize=None)
def signs_zero():
    """Every pair of the special values on (x, y) and on (y, z); the third axis holds a separator voxel per pair of
    magnitude classes, so that no voxel mixes denormals, 1e-30 and leaf-sized values (their fp64 sums stay exact)."""
    leaf = 0.01
    rng = np.random.default_rng(5)
    sv = signs_zero_values(leaf)
    rows = []
    for a, ca in sv:
        for b, cb in sv:
            sep = float(solve(np.array([3 * (3 * ca + cb) + 2]), leaf)[0])
            for _ in range(2):
                rows.append((a, b, sep))
                rows.append((sep, a, b))
    p = np.array(rows, dtype=f32)
    return Case(points(p[rng.permutation(len(p))], rng), leaf)


@functools.lru_cache(maxsize=None)
def far_keys(leaf):
    """Indices at +-2^20 (+-1), pairs of voxels 2^21 * k cells apart on one axis (all three axes for some), and
    coordinates whose product with 1/leaf passes +-2^31, up to +-FLT_MAX (saturated to INT_MAX / INT_MIN)."""
    rng = np.random.default_rng(int(1 / leaf))
    rows, pairs = [], []
    for t in (2 ** 20 - 1, 2 ** 20, 2 ** 20 + 1, -(2 ** 20 - 1), -(2 ** 20), -(2 ** 20 + 1)):
        for d in range(3):
            idx = np.array([[3, -4, 5]] * 2)
            idx[:, d] = t
            rows.append(in_voxels(idx, leaf, rng))
    inv = np.float64(inv_leaf(leaf))
    for d in range(3):
        for k in (1, 2, 3, -1, -2, -7, 100, -100, 1000, -1023, 1023):
            target = int(rng.integers(-500, 500)) + k * 2 ** 21
            x2 = f32(target / inv)
            i2 = int(voxel_index(x2, leaf))
            i1 = i2 - k * 2 ** 21
            other = rng.integers(-50, 50, 3)
            a = np.array([other, other])
            a[0, d] = i1
            pa = in_voxels(a[:1], leaf, rng)
            pb = in_voxels(a[:1], leaf, rng)
            far = pa.copy()
            far[0, d] = x2
            rows += [pa, pb, far]
            pairs.append((i1, i2))
        # 2^21 apart on all three axes at once
        i1 = rng.integers(-500, 500, 3)
        near = in_voxels(i1[None, :], leaf, rng)
        far3 = np.stack([f32((i1[e] + 2 ** 21 * (d + 1)) / inv) for e in range(3)])[None, :]
        rows += [near, far3]
    # saturation: products past +-2^31 on each axis; a voxel mixing magnitudes holds two points, one of a kind more
    edge = f32(2.0 ** 31 / inv)
    sat = [2.2e9 / inv, 1e30, 3e38, F32_MAX, float(edge), float(ulps(edge, -1)), -2.2e9 / inv, -1e30, -3e38, -F32_MAX,
           float(-edge), float(ulps(-edge, 1)), float(ulps(-edge, -1))]
    for d in range(3):
        for j, v in enumerate(sat):
            idx = np.array([[j + 60] * 3])
            p = in_voxels(idx, leaf, rng)
            p[0, d] = v
            rows.append(p)
        for g, group in enumerate(((2.2e9 / inv, 3e38), (3e38, F32_MAX, 1e38), (-1e30, -3e38))):
            idx = np.array([[40 + g] * 3])
            base = in_voxels(idx, leaf, rng)
            for v in group:
                p = base.copy()
                p[0, d] = v
                rows.append(p)
    p = np.concatenate(rows).astype(f32)
    c = Case(points(p, rng), leaf)
    c.pairs = pairs
    return c


@functools.lru_cache(maxsize=None)
def own_voxels(n):
    """n = capacity points, each in a voxel of its own, in random order."""
    rng = np.random.default_rng(n)
    v = rng.permutation(n)
    idx = np.stack([v % 100 + 10, (v // 100) % 100 - 150, v // 10000 + 20], axis=1)
    return Case(points(in_voxels(idx, 0.01, rng), rng), 0.01)


@functools.lru_cache(maxsize=None)
def one_voxel():
    """300 000 points in voxel (50, 50, 150): colour sums pass 2^24, all points hit one hash slot."""
    rng = np.random.default_rng(3)
    n = 300000
    p = f32([0.5, 0.5, 1.5]) + rng.uniform(0.0005, 0.0095, (n, 3)).astype(f32)
    rgba = (rng.integers(200, 256, (n, 3)) * [1 << 16, 1 << 8, 1]).sum(axis=1).astype(np.uint32)
    return Case(oracle.make_points(p, rgba), 0.01)


CHAIN_CAPS = [512, 513, 4096, 4097]


@functools.lru_cache(maxsize=None)
def chain(cap):
    """n = cap points: 320 voxels whose hash homes them all on slot H - 5 of the H-slot table (the probe chain runs
    off the end of the table and wraps to slot 0), some with a second point, the rest elsewhere."""
    rng = np.random.default_rng(cap)
    H = table_size(cap)
    home = np.uint64(H - 5)
    found = []
    for z0 in range(10, 10000, 16):
        g = np.stack(np.meshgrid(np.arange(-128, 128), np.arange(-128, 128), np.arange(z0, z0 + 16), indexing="ij"), -1).reshape(-1, 3)
        found.append(g[(voxel_hash(g[:, 0], g[:, 1], g[:, 2]) & np.uint64(H - 1)) == home])
        if sum(len(f) for f in found) >= 320:
            break
    hot = np.concatenate(found)[:320]
    dup = min(320, cap - 400)  # a second point in as many chained voxels as the capacity leaves room for
    m = cap - 320 - dup
    idx = np.concatenate([hot, hot[:dup], np.stack([rng.integers(300, 400, m), rng.integers(-50, 50, m), rng.integers(-50, 50, m)], 1)])
    idx = idx[rng.permutation(cap)]
    c = Case(points(in_voxels(idx, 0.01, rng), rng), 0.01)
    c.hot = hot
    return c


@functools.lru_cache(maxsize=None)
def random_cloud(n):
    """n = capacity points in a 2 m cube away from the coordinate planes, a few per voxel, 5 % NaN."""
    rng = np.random.default_rng(n)
    p = rng.uniform(0.5, 1.1, (n, 3)).astype(f32)
    p[rng.random(n) < 0.05, rng.integers(0, 3)] = np.nan
    return Case(points(p, rng), 0.01, 2, 0.6, 1.05)


def tile_edges(n):
    e = [t * TILE + o for t in range(1, n // TILE + 1) for o in (-1, 0)]
    return sorted({i for i in e + [n - 1] if 0 <= i < n})


@functools.lru_cache(maxsize=None)
def tiled(n):
    """n points, z limits [0, 10]: a fresh voxel first appears exactly at every tile edge t * 4096 - 1, t * 4096 and
    at n - 1; the points right beside each edge are rejected (NaN in one coordinate, or z outside the limits) and lie
    in fresh voxels too.  Everything else falls in a pool of voxels that appear in random order."""
    rng = np.random.default_rng(n + 17)
    first = tile_edges(n)
    reject = sorted({i for t in range(1, n // TILE + 1) for i in (t * TILE - 2, t * TILE + 1)} - set(first))
    reject = [i for i in reject if 0 <= i < n]
    idx = np.stack([rng.integers(10, 12 + n // 384, n), rng.integers(-4, 4, n), rng.integers(100, 108, n)], axis=1)
    fresh = np.stack([-20 - np.arange(len(first) + len(reject)), np.zeros(len(first) + len(reject), np.int64),
                      np.full(len(first) + len(reject), 500)], axis=1)
    special = np.array(first + reject, np.int64)
    idx[special] = fresh
    later = rng.integers(0, n, len(first))  # later points of the fresh voxels (after their first one)
    taken = set(special.tolist())
    for f, j in zip(first, later):
        if j > f and j not in taken:
            idx[j] = idx[f]
    p = in_voxels(idx, 0.01, rng)
    for k, i in enumerate(reject):
        if k % 3 == 0:
            p[i, k % 2] = np.nan
        else:
            p[i, 2] = f32(-0.5) if k % 2 else f32(10.5)
    c = Case(points(p, rng), 0.01, 2, 0.0, 10.0)
    c.first, c.reject = first, reject
    return c


TILED_N = [4095, 4097, 8191, 8193, 3 * TILE + 7, 4194305, 5000011]

LIMIT_VALUES = [-0.5, 0.25, 0.3, 1.0, 0.5, 0.0]
LIMITS = [(0, -0.5, 0.25), (1, 0.3, 0.3), (2, 1.0, 0.5), (2, -np.inf, np.inf), (0, -np.inf, 0.0), (1, 0.0, np.inf), (2, np.nan, 1.0),
          (0, -0.5, np.nan), (1, np.nan, np.nan), (-1, 0.0, 0.0)]


@functools.lru_cache(maxsize=None)
def limit_cloud():
    """Coordinates at every limit value and 1-2 ulp either side, NaN and +-inf, in random triples."""
    rng = np.random.default_rng(23)
    vals = np.concatenate([ulps([v], s) for v in LIMIT_VALUES for s in (0, 1, -1, 2, -2)] + [f32([np.nan, np.inf, -np.inf])])
    finite = vals[np.isfinite(vals)]
    p = finite[rng.integers(0, len(finite), (6000, 3))]
    odd = rng.random((6000, 3)) < 0.03
    p[odd] = vals[rng.integers(len(vals) - 3, len(vals), odd.sum())]
    return points(p, rng)


def limit_case(k):
    field, lo, hi = LIMITS[k]
    return Case(limit_cloud(), 0.01, field, lo, hi)


ZERO_VALUES = [f32(0.01), np.nextafter(f32(0.01), f32(0)), np.nextafter(f32(0.01), f32(1)), ulps(f32(0.01), 2), f32(-0.01),
               np.nextafter(f32(-0.01), f32(0)), np.nextafter(f32(-0.01), f32(-1)), f32(0.0), f32(-0.0), f32(0.5), f32(0.00999), f32(-0.3)]


@functools.lru_cache(maxsize=None)
def zero_cloud():
    """Every triple of values at |c| = 0.01f and its neighbours (0.01f < 0.01 in double: such a point is removed), plus
    a few non-finite points."""
    rng = np.random.default_rng(31)
    z = np.array(ZERO_VALUES, dtype=f32)
    g = np.stack(np.meshgrid(z, z, z, indexing="ij"), -1).reshape(-1, 3)
    g = g[rng.permutation(len(g))]
    g[rng.choice(len(g), 20, replace=False), rng.integers(0, 3)] = np.nan
    g[rng.choice(len(g), 5, replace=False), 1] = np.inf
    return points(g, rng)


def remove_zero_reference(pts):
    p = xyz(pts).astype(np.float64)
    return pts[np.isfinite(p).all(axis=1) & ~(np.abs(p) < 0.01).all(axis=1)]


CASES = {"lattice": (lattice, [(l,) for l in LATTICE_LEAVES]), "signs_zero": (signs_zero, [()]),
         "far_keys": (far_keys, [(0.01,), (0.001,), (1e-4,)]), "own_voxels": (own_voxels, [(100000,)]), "one_voxel": (one_voxel, [()]),
         "chain": (chain, [(c,) for c in CHAIN_CAPS]), "random": (random_cloud, [(512,), (513,), (65536,), (65537,), (2 ** 20,), (2 ** 20 + 1,)]),
         "tiled": (tiled, [(n,) for n in TILED_N]), "limits": (limit_case, [(k,) for k in range(len(LIMITS))])}
ALL = [(name, args) for name, (_, arglist) in CASES.items() for args in arglist]
IDS = ["%s%s" % (name, "-" + "-".join(str(a) for a in args) if args else "") for name, args in ALL]


def case(name, args):
    return CASES[name][0](*args)


@functools.lru_cache(maxsize=4)
def ref_of(name, args):
    c = case(name, args)
    return reference(c.pts, c.leaf, c.field, c.lo, c.hi, with_free=True)


# ------------------------------------------------------------------ CPU: every case has its property
@pytest.mark.parametrize("name,args", ALL, ids=IDS)
def test_case_sums_are_order_free_and_oracle_agrees(name, args):
    """Every voxel's fp64 sums are exact in any order (so the GPU's atomics cannot change a bit), and the C++ oracle
    gives the reference's points bit for bit."""
    c = case(name, args)
    want, free = ref_of(name, args)
    assert len(want) > 0 or name == "limits"
    assert free.all(), "%d voxels whose fp64 sums depend on the order" % (~free).sum()
    assert_same(oracle.voxel_grid_exact(c.pts, c.leaf, c.field, c.lo, c.hi), want)


@pytest.mark.parametrize("leaf", LATTICE_LEAVES)
def test_lattice_has_faces_where_product_and_division_disagree(leaf):
    c = lattice(leaf)
    p = xyz(c.pts)
    prod = p * inv_leaf(leaf)
    assert (prod == np.floor(prod)).sum() > 1000  # exactly on a face of the fp32 lattice
    exact = np.floor(p.astype(np.float64) / np.float64(f32(leaf)))
    disagree = (voxel_index(p, leaf) != exact).any(axis=1)
    assert disagree.sum() > 100
    if leaf == 0.01:
        k = np.arange(-3000, 3000).astype(f32) * f32(0.01)
        assert (voxel_index(k, 0.01) != np.floor(k.astype(np.float64) / np.float64(f32(0.01)))).sum() == 2341
        assert voxel_index(f32(-30.0), 0.01) == -3000
    want = ref_of("lattice", (leaf,))[0]
    assert len(want) < len(c.pts) - 1000  # voxels on a face hold points from both sides


def test_signs_zero_sums_are_exact_in_input_order():
    c = signs_zero()
    p = xyz(c.pts)
    keys = np.stack([voxel_index(p[:, d], c.leaf) for d in range(3)], axis=1)
    ids, _ = voxel_ids(keys)
    for d in range(3):
        seq = np.bincount(ids, weights=p[:, d].astype(np.float64))
        exact = np.array([math.fsum(p[ids == k, d].astype(np.float64)) for k in range(ids.max() + 1)])
        assert np.array_equal(seq, exact)
    assert set(np.unique(keys).tolist()) >= {-1, 0}
    assert (np.signbit(p) & (p == 0)).any() and ((p != 0) & (np.abs(p) < 2.0 ** -126)).any()
    assert np.bincount(ids).max() >= 3


@pytest.mark.parametrize("leaf", [0.01, 0.001, 1e-4])
def test_far_keys_reach_the_int32_edges_and_share_21_bit_residues(leaf):
    c = far_keys(leaf)
    p = xyz(c.pts)
    keys = np.stack([voxel_index(p[:, d], leaf) for d in range(3)], axis=1)
    for t in (2 ** 20 - 1, 2 ** 20, 2 ** 20 + 1):
        assert (keys == t).any() and (keys == -t).any()
    assert (keys == I32_MAX).any() and (keys == I32_MIN).any()
    assert (np.abs(p.astype(np.float64) * np.float64(inv_leaf(leaf))) >= 2.0 ** 31).sum() >= 30
    for i1, i2 in c.pairs:
        assert i1 != i2 and (i2 - i1) % 2 ** 21 == 0 and abs(i1) < 2 ** 20
    # the 21-bit packing of the parent commit's key gives these distinct voxels one key
    packed = (keys + 2 ** 20) & 0x1fffff
    assert len(np.unique(packed, axis=0)) < len(np.unique(keys, axis=0)) - 30


@pytest.mark.parametrize("cap", CHAIN_CAPS)
def test_chain_shares_one_home_slot_and_wraps(cap):
    c = chain(cap)
    assert len(c.pts) == cap
    H = table_size(cap)
    assert H == (1024 if cap <= 512 else 2048 if cap <= 1024 else 8192 if cap <= 4096 else 16384)
    keys = np.stack([voxel_index(xyz(c.pts)[:, d], 0.01) for d in range(3)], axis=1)
    uk = np.unique(keys, axis=0)
    home = voxel_hash(uk[:, 0], uk[:, 1], uk[:, 2]) & np.uint64(H - 1)
    assert (home == H - 5).sum() >= 300
    # linear probing in any insertion order: the chain holds every key homed at H - 5, so it runs past slot H - 1
    table = np.full(H, -1, np.int64)
    for k, h in enumerate(home.astype(np.int64)):
        s = h
        while table[s] >= 0:
            s = (s + 1) % H
        table[s] = k
    assert (table[:300] >= 0).all()


@pytest.mark.parametrize("n", TILED_N)
def test_tiled_first_points_sit_on_tile_edges(n):
    c = tiled(n)
    assert len(c.pts) == n
    ok = passes(c.pts, c.field, c.lo, c.hi)
    p = xyz(c.pts)[ok]
    keys = np.stack([voxel_index(p[:, d], c.leaf) for d in range(3)], axis=1)
    _, first = voxel_ids(keys)
    first_in = set(np.flatnonzero(ok)[first].tolist())
    assert set(c.first) <= first_in and n - 1 in first_in
    assert not ok[c.reject].any()
    if n > 1024 * TILE:
        assert -(-n // TILE) > 1024  # more tiles than one pass of the tile scan takes
    assert len(first_in) > 1


def test_limits_and_zero_points_cover_their_edges():
    pts = limit_cloud()
    p = xyz(pts)
    for field, lo, hi in LIMITS:
        ok = passes(pts, field, lo, hi)
        if field >= 0 and np.isfinite(lo) and np.isfinite(hi) and lo <= hi:
            v = p[:, field]
            assert ((v == f32(lo)) & ok).any() and ((v == f32(hi)) & ok).any()
            assert ((v == np.nextafter(f32(lo), f32(-np.inf))) & ~ok).any()
    assert passes(pts, 2, 1.0, 0.5).sum() == 0 and passes(pts, 1, 0.3, 0.3).sum() > 0
    assert np.isnan(p[~np.isfinite(p).all(axis=1)]).any() and np.isinf(p).any()
    z = zero_cloud()
    kept = remove_zero_reference(z)
    c = f32(0.01)
    assert float(c) < 0.01
    triple = (z["x"] == c) & (z["y"] == c) & (z["z"] == c)
    assert triple.sum() == 1 and not ((kept["x"] == c) & (kept["y"] == c) & (kept["z"] == c)).any()
    up = np.nextafter(c, f32(1))
    assert ((kept["x"] == up) & (kept["y"] == up) & (kept["z"] == up)).sum() == 1


# ------------------------------------------------------------------ GPU
def gpu_voxel_grid(cloud, leaf, field, lo, hi, out=None):
    vg = pcl.VoxelGrid()
    vg.setLeafSize(leaf)
    vg.setPassThrough(None if field < 0 else "xyz"[field], lo, hi)
    vg.setInputCloud(cloud)
    return vg.filter(out)


@pytest.mark.gpu
@pytest.mark.parametrize("name,args", ALL, ids=IDS)
def test_voxel_grid_matches_reference(name, args):
    c = case(name, args)
    want, free = ref_of(name, args)
    assert free.all()
    assert_same(gpu_voxel_grid(pcl.PointCloud(c.pts), c.leaf, c.field, c.lo, c.hi).to_numpy(), want)


@pytest.mark.gpu
@pytest.mark.parametrize("leaf", [0.01, 0.001, 1e-4])
def test_far_keys_through_pcl_approximate_voxel_grid(leaf):
    """upstream's 512-slot cache on the same coordinates: saturated indices and the unsigned 7171 / 3079 / 4231 hash"""
    c = far_keys(leaf)
    fin = c.pts[np.isfinite(xyz(c.pts)).all(axis=1)]
    want = oracle.approx_voxel_grid_pcl(fin, leaf)
    vg = pcl.VoxelGrid()
    vg.setLeafSize(leaf)
    vg.setPclApproximateMode(True)
    vg.setInputCloud(pcl.PointCloud(c.pts))
    got = vg.filter().to_numpy()
    assert len(got) == len(want) and np.array_equal(bits(got), bits(want))


@pytest.mark.gpu
@pytest.mark.parametrize("k", range(len(LIMITS)))
def test_passthrough_limits(k):
    field, lo, hi = LIMITS[k]
    if field < 0:
        return
    pts = limit_cloud()
    pt = pcl.PassThrough()
    pt.setFilterFieldName("xyz"[field])
    pt.setFilterLimits(lo, hi)
    pt.setInputCloud(pcl.PointCloud(pts))
    got = pt.filter().to_numpy()
    want = pts[passes(pts, field, lo, hi)]
    assert len(got) == len(want) and np.array_equal(bits(got), bits(want))


@pytest.mark.gpu
def test_remove_zero_points_and_prepare_model_at_one_centimetre():
    z = zero_cloud()
    want = remove_zero_reference(z)
    got = pcl.removeZeroPoints(pcl.PointCloud(z)).to_numpy()
    assert len(got) == len(want) and np.array_equal(bits(got), bits(want))
    model, c = pcl.prepare_model(pcl.PointCloud(z), 0.01)
    w = xyz(want).astype(np.float64)
    centroid = np.array([math.fsum(w[:, d]) for d in range(3)]) / len(w)
    assert np.array_equal(np.asarray(c, f32).view(np.uint32), centroid.astype(f32).view(np.uint32))
    moved = want.copy()
    for d, k in enumerate("xyz"):
        moved[k] = want[k] - f32(c[d])
    ref, free = reference(moved, 0.01, with_free=True)
    assert free.all()
    assert_same(model.to_numpy(), ref)


def _qhd_cameras():
    rng = np.random.default_rng(8)
    cams = []
    for k in range(8):
        depth = rng.integers(500, 4500, (540, 960)).astype(np.uint16)
        depth[rng.random((540, 960)) < 0.02] = 0
        a = k * np.pi / 4
        pose = np.eye(4)
        pose[:2, :2] = [[np.cos(a), -np.sin(a)], [np.sin(a), np.cos(a)]]
        pose[:3, 3] = [10.0 + 0.01 * k, 10.0, 10.0]
        cams.append(dict(depth=depth, bgr=rng.integers(0, 256, (540, 960, 3), dtype=np.uint8), fx=540.0, fy=540.0, cx=479.5, cy=269.5, pose=pose))
    return cams


@pytest.mark.gpu
def test_eight_fused_qhd_cameras():
    """8 x 960 x 540 = 4 147 200 points, just under 1024 tiles, fused on the device, then downsampled."""
    fused = pcl.PointCloud().fromDepthImages(_qhd_cameras())
    pts = fused.to_numpy()
    assert len(pts) == 8 * 960 * 540
    want, free = reference(pts, 0.01, 2, 0.0, 20.0, with_free=True)
    assert free.all() and len(want) > 100000
    assert_same(gpu_voxel_grid(fused, 0.01, 2, 0.0, 20.0).to_numpy(), want)


def _graph_cloud():
    rng = np.random.default_rng(77)
    c = lattice(0.01).pts
    extra = points(np.array([[0.5, 0.5, 10.0], [0.5, 0.5, 1.0], [1.0, -1.0, 0.5], [-1.0, 0.25, 0.25]] * 3, dtype=f32), rng)
    return np.concatenate([c[:20000], extra])


GRAPH_CONFIGS = [(0.01, 2, 0.0, 10.0), (0.02, 2, 0.0, 10.0), (0.01, 2, 0.0, 10.0), (0.01, 2, 1.0, 10.0), (0.01, 0, -1.0, 1.0),
                 (0.01, -1, 0.0, 0.0), (float(np.nextafter(f32(0.01), f32(1))), 2, 0.0, 10.0), (0.01, 2, 0.0, float(np.nextafter(f32(10), f32(0)))),
                 (0.01, 1, -1.0, 1.0), (0.01, 2, 0.0, 10.0)]


def test_graph_configs_change_the_result():
    """Each change of leaf (by one ulp too), limits or field between calls on one pair changes the downsample, so a
    stale graph cannot pass; the first configuration comes back twice (replays of its graph)."""
    pts = _graph_cloud()
    seen = [bits(reference(pts, *c)).tobytes() for c in GRAPH_CONFIGS]
    assert len(set(seen)) == len(GRAPH_CONFIGS) - 2 and seen[0] == seen[2] == seen[-1]


@pytest.mark.gpu
def test_graph_cache_one_pair_changing_parameters():
    pts = _graph_cloud()
    cloud, out = pcl.PointCloud(pts), pcl.PointCloud()
    for leaf, field, lo, hi in GRAPH_CONFIGS:
        assert_same(gpu_voxel_grid(cloud, leaf, field, lo, hi, out).to_numpy(), reference(pts, leaf, field, lo, hi))


@pytest.mark.gpu
def test_graph_cache_double_buffered_async_frames():
    """Ten frames of different sizes uploaded asynchronously, alternately into two clouds, the next upload enqueued
    before the current frame is downsampled; then the same frames through a PassThrough into one cloud of fixed
    capacity, whose point count changes under a cached graph."""
    rng = np.random.default_rng(91)
    base = random_cloud(65536).pts
    sizes = [5000, 7000, 3000, 7000, 12000, 1, 9000, 4096, 4097, 7000]
    frames = [base[rng.permutation(len(base))[:n]] for n in sizes]
    bufs = [pcl.PinnedBuffer.of(f) for f in frames]
    clouds, outs = [pcl.PointCloud(), pcl.PointCloud()], [pcl.PointCloud(), pcl.PointCloud()]
    clouds[0].upload_raw_async(bufs[0].ptr, sizes[0])
    for k in range(10):
        if k + 1 < 10:
            clouds[(k + 1) % 2].upload_raw_async(bufs[k + 1].ptr, sizes[k + 1])
        got = gpu_voxel_grid(clouds[k % 2], 0.01, 2, 0.6, 1.05, outs[k % 2]).to_numpy()
        assert_same(got, reference(frames[k], 0.01, 2, 0.6, 1.05))
    big = pcl.PointCloud(base)
    mid, out = pcl.PointCloud(), pcl.PointCloud()
    pt = pcl.PassThrough()
    pt.setFilterFieldName("x")
    pt.setInputCloud(big)
    for k in range(10):
        hi = 0.5 + 0.06 * (k + 1) * (1 if k % 3 else 0.5)
        pt.setFilterLimits(0.5, hi)
        pt.filter(mid)
        sub = base[passes(base, 0, 0.5, hi)]
        assert_same(gpu_voxel_grid(mid, 0.01, 2, 0.6, 1.05, out).to_numpy(), reference(sub, 0.01, 2, 0.6, 1.05))


@pytest.mark.gpu
def test_graph_cache_more_pairs_than_graphs():
    """Ten (in, out) pairs in rotation, three rounds (every graph evicted and captured again), new contents each round;
    then four pairs (cached graphs replayed) with new contents."""
    rng = np.random.default_rng(5)
    base = random_cloud(65536).pts
    ins, outs = [pcl.PointCloud() for _ in range(10)], [pcl.PointCloud() for _ in range(10)]
    for r in range(4):
        pairs = range(10) if r < 3 else range(4)
        for _ in range(1 if r < 3 else 2):
            for k in pairs:
                frame = base[rng.permutation(len(base))[:3000 + 100 * k]]
                ins[k].upload(frame)
                assert_same(gpu_voxel_grid(ins[k], 0.01, 2, 0.6, 1.05, outs[k]).to_numpy(), reference(frame, 0.01, 2, 0.6, 1.05))
