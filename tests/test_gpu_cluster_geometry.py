"""Euclidean cluster extraction on adversarial geometry, against a brute-force neighbour graph.

A cluster is a connected component of the graph "fp32 d2 < (float)(tolerance^2)", d2 = (dx*dx + dy*dy) + dz*dz with
every operation rounded (PCL's KdTree radius search).  Both the GPU (pft_cluster.cu) and the oracle serve that search
from a uniform grid, so a grid that misses a pair is invisible when one is compared with the other.  The reference here
shares nothing with either grid: candidate pairs come from scipy's kd-tree at radius tol * (1 + 1e-4) in fp64 (a strict
superset of the fp32 predicate: a pair that passes it is at most tol * (1 + 2^-22) apart), the fp32 predicate is applied
to each, and scipy's connected components give the clusters.  Exact duplicates (d2 = 0) are joined to their first copy
instead of being listed pairwise.

The cases, each built for one way the extraction can go wrong:

  boundary     pairs along x, y, z and diagonals whose fp32 d2 is pred(T), T and succ(T), T = (float)(tol^2), for
               tolerances where (float)(tol^2) and (float)tol * (float)tol agree and where they do not
  long grids   the three-point witness, bead chains spaced just under the tolerance along 80 m, 400 m and 2000 m lines
               and inside thin slabs, and pairs that straddle two cells under the former fp32 cell formula
  cell size    clouds whose extent forces a cell larger than the tolerance (the former loop doubled it 1, 9, 33 times)
  extremes     tolerance 1e-15, points at +-1e13 and +-3e38, two finite singletons, NaN and +-inf in one coordinate
               (the former sizing loop fell through for several of them and left the cell count unset)
  union-find   chains whose indices run against the geometry, two zipped chains, a permuted 100 k-point surface, 10 k
               copies of one point and a 200 k-point component; every GPU case is extracted twice
  selection    sizes at min and max, min == max, equal-size ties, singletons, exactly 4096 passing clusters (the select
               kernel's sort holds 4096) and 4097 (PFT_ERR_CAPACITY), a cluster spread over several 4096-point scan tiles

The tests without the gpu mark compare the oracle with the reference and check on the CPU that each case has the
property it was built for; the gpu tests compare EuclideanClusterExtraction with the reference: sizes, labels and every
cluster_cloud(k) bit for bit."""
import functools

import numpy as np
import pytest
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components
from scipy.spatial import cKDTree

import oracle
from pcl_tracking_b200 import pcl, synth

f32 = np.float32
MAX_CLUSTERS = 4096      # kMaxClusters: clusters that can pass the size filter
MAX_CELLS = 1 << 22      # kMaxClusterCells
BIG = 2 ** 31 - 1


class Case:
    def __init__(self, xyz, tol, mn=1, mx=BIG, rgba_seed=0, **props):
        xyz = np.asarray(xyz, dtype=f32).reshape(-1, 3)
        rng = np.random.default_rng(rgba_seed)
        self.pts = oracle.make_points(xyz, rng.integers(0, 1 << 32, len(xyz), dtype=np.uint64).astype(np.uint32))
        self.xyz, self.tol, self.mn, self.mx, self.props = xyz, tol, mn, mx, props


def d2_f32(a, b):
    """PCL's fp32 squared distance, every operation rounded."""
    with np.errstate(over="ignore", invalid="ignore"):
        d = (np.asarray(a, f32) - np.asarray(b, f32)).astype(f32)
        return ((d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]).astype(f32)


def t2_of(tol):
    return f32(tol * tol)  # KdTreeFLANN::radiusSearch: (float)(radius * radius)


# ------------------------------------------------------------------ the reference
def reference(xyz, tol, mn, mx):
    """(labels, sizes, edges): the clusters of the brute-force neighbour graph in ec.labels / ec.sizes form (size
    descending, then lowest member index ascending) and the joined pairs as original point indices."""
    n = len(xyz)
    fin = np.flatnonzero(np.isfinite(xyz).all(axis=1))
    P = xyz[fin]
    m = len(P)
    t2 = t2_of(tol)
    _, rep, inv = np.unique(np.ascontiguousarray(P).view(np.uint32).reshape(m, 3), axis=0, return_index=True, return_inverse=True)
    inv = inv.reshape(-1)
    a_list, b_list = [], []
    if t2 > 0:                                  # exact copies: d2 = 0
        dup = rep[inv] != np.arange(m)
        a_list.append(np.flatnonzero(dup)); b_list.append(rep[inv][dup])
    U = P[rep]
    pairs = cKDTree(U.astype(np.float64)).query_pairs(tol * (1 + 1e-4), output_type="ndarray")
    assert len(pairs) < 10_000_000
    if len(pairs):
        keep = d2_f32(U[pairs[:, 0]], U[pairs[:, 1]]) < t2
        a_list.append(rep[pairs[keep, 0]]); b_list.append(rep[pairs[keep, 1]])
    a = np.concatenate(a_list) if a_list else np.zeros(0, np.int64)
    b = np.concatenate(b_list) if b_list else np.zeros(0, np.int64)
    g = coo_matrix((np.ones(len(a), np.int8), (a, b)), shape=(m, m))
    nc, comp = connected_components(g, directed=False)
    size = np.bincount(comp, minlength=nc)
    low = np.full(nc, m, dtype=np.int64)
    np.minimum.at(low, comp, np.arange(m))     # fin is ascending: the lowest member in input order
    ok = np.flatnonzero((size >= mn) & (size <= mx))
    order = ok[np.lexsort((low[ok], -size[ok]))]
    rank = np.full(nc, -1, dtype=np.int32)
    rank[order] = np.arange(len(order), dtype=np.int32)
    labels = np.full(n, -1, dtype=np.int32)
    labels[fin] = rank[comp]
    return labels, size[order].astype(np.int32), np.stack([fin[a], fin[b]], axis=1)


# ------------------------------------------------------------------ grid restatements
def prefix_grid(xyz, tol):
    """RESTATEMENT OF THE FORMER (PRE-FIX) GRID of pft_cluster.cu, fp32 without FMA: origin = the bounding box minimum,
    cell = (float)tol * 1.0001f doubled at most 40 times until the grid has <= 2^22 cells, cell coordinate
    floorf((x - origin) * (1 / cell)).  Returns (doublings or None when the loop falls through, origin, inv_cell, dims)."""
    fin = np.isfinite(xyz).all(axis=1)
    lo, hi = xyz[fin].min(axis=0), xyz[fin].max(axis=0)
    c = f32(f32(tol) * f32(1.0001))
    with np.errstate(over="ignore"):
        for it in range(40):
            cells, dims = 1, []
            for d in range(3):
                dims.append(int(min(np.floor(f32(f32(hi[d] - lo[d]) / c)), f32(2.0e9))) + 1)
                cells = min(cells * dims[-1], 1 << 40)
            if cells <= MAX_CELLS:
                return it, lo, f32(1.0) / c, dims
            c = f32(c * f32(2.0))
    return None, lo, f32(1.0) / c, dims


def prefix_cells(xyz, tol):
    it, lo, inv, dims = prefix_grid(xyz, tol)
    assert it is not None
    with np.errstate(invalid="ignore"):
        s = np.floor(((xyz - lo).astype(f32) * inv).astype(f32))
    return np.clip(np.nan_to_num(s), 0, np.array(dims) - 1).astype(np.int64)


def fixed_cells(xyz, tol):
    """The grid of pft_cluster.cu as it is now, restated in fp64: (cells of every point, dims)."""
    fin = np.isfinite(xyz).all(axis=1)
    lo, hi = xyz[fin].min(axis=0).astype(np.float64), xyz[fin].max(axis=0).astype(np.float64)
    L = hi - lo
    q = float((MAX_CELLS - 1) // 3)
    c = tol * 1.0001
    c = max(c, (L[0] + L[1] + L[2]) / q)
    c = max(c, float(np.sqrt((L[0] * L[1] + L[0] * L[2] + L[1] * L[2]) / q)))
    c = max(c, float(np.cbrt(L[0] * L[1] * L[2] / q)))
    c *= 1.0 + 2.0 ** -20
    dims = np.floor(L / c).astype(np.int64) + 1
    with np.errstate(invalid="ignore"):
        s = np.floor((xyz.astype(np.float64) - lo) / c)
    return np.clip(np.nan_to_num(s), 0, dims - 1).astype(np.int64), dims


def straddles(cells, edges):
    """Joined pairs whose cells are more than one apart on some axis: pairs a 27-cell neighbourhood never compares."""
    return np.flatnonzero((np.abs(cells[edges[:, 0]] - cells[edges[:, 1]]) > 1).any(axis=1))


# ------------------------------------------------------------------ builders
def boundary_case(tol):
    """Isolated pairs whose fp32 d2 is pred(T), T and succ(T) (each where the direction can reach it; otherwise the nearest
    d2 on each side of T), along x, y, z and the four diagonals.  Each pair starts at a base point whose moving
    coordinates are 0 (1/16 for the xyz diagonal), so the differences are exact; the k-th pair of a direction is moved
    0.25 k m along a coordinate that is equal within the pair (the xyz diagonal: along z, and searched again there)."""
    T = t2_of(tol)
    targets = (np.nextafter(T, f32(0)), T, np.nextafter(T, f32(np.inf)))
    fams = [((1, 0, 0), (0.0, 2.0, 3.0), 1), ((0, 1, 0), (3.0, 0.0, 2.0), 2), ((0, 0, 1), (2.0, 3.0, 0.0), 0),
            ((1, 1, 0), (0.0, 0.0, 5.0), 2), ((0, 1, 1), (5.0, 0.0, 0.0), 0), ((1, 0, 1), (0.0, 5.0, 0.0), 1),
            ((1, 1, 1), (0.0625, 0.0625, 0.0625), 2)]
    out, found = [], set()
    for direction, base0, far in fams:
        u = np.array(direction, np.float64) / np.linalg.norm(direction)
        seen = set()
        for k in range(5):   # pred(T), T, succ(T), the largest d2 below T, the smallest d2 from T up
            base = np.array(base0, f32)
            base[far] += f32(0.25 * k)
            b0 = (base + u * np.sqrt(float(T))).astype(f32)
            axes = [b0[d] + np.arange(-12, 13) * np.abs(np.spacing(b0[d])) if direction[d] else np.array([b0[d]]) for d in range(3)]
            B = np.stack(np.meshgrid(*axes, indexing="ij"), axis=-1).reshape(-1, 3).astype(f32)
            d2 = d2_f32(np.broadcast_to(base, B.shape), B)
            if k < 3:
                hit = np.flatnonzero(d2 == targets[k])
                if not len(hit):
                    continue
                p = hit[0]
            else:
                side = np.flatnonzero(d2 < T) if k == 3 else np.flatnonzero(d2 >= T)
                p = side[np.argmax(d2[side])] if k == 3 else side[np.argmin(d2[side])]
            if float(d2[p]) in seen:
                continue
            seen.add(float(d2[p]))
            out += [base, B[p]]
        found |= seen
    return Case(np.array(out), tol, boundary_targets=[float(t) for t in targets], found=found)


def walk_below(prev, nxt, axis, T):
    """Move nxt[:, axis] (above prev) down until the fp32 d2 to prev is below T, one step at a time: an ulp of the
    coordinate or of the difference, whichever is larger (both are powers of two, so the step is exact)."""
    while True:
        bad = np.flatnonzero(d2_f32(prev, nxt) >= T)
        if not len(bad):
            return nxt
        x = nxt[bad, axis]
        step = np.maximum(np.abs(np.spacing(x)), np.spacing((x - prev[bad, axis]).astype(f32)))
        nxt[bad, axis] = (x - step).astype(f32)


def chains_case(length, tol, axis, origin, slab=None, beads=8, seed=0):
    """n_chains bead chains along `axis`, each bead as far from the previous one as the fp32 predicate allows, laid out
    over `length` metres from an unround origin; two anchor points set the bounding box.  With `slab` = (w1, w2) the
    chains are spread over a slab of that cross-section instead of one line."""
    rng = np.random.default_rng(seed)
    T = t2_of(tol)
    other = [d for d in range(3) if d != axis]
    n_chains = min(400, int(length / ((beads + 4) * tol)) - 1)
    pitch = length / (n_chains + 1)
    start = np.zeros((n_chains, 3), np.float64)
    start[:, axis] = origin[axis] + pitch * (np.arange(n_chains) + 0.5) + rng.uniform(0, pitch - (beads + 2) * tol, n_chains)
    for k, d in enumerate(other):
        w = 0.0 if slab is None else slab[k]
        start[:, d] = origin[d] + rng.uniform(0, w, n_chains)
    cur = start.astype(f32)
    pts = [cur]
    for _ in range(beads - 1):
        nxt = cur.copy()
        nxt[:, axis] = (cur[:, axis] + f32(tol)).astype(f32)
        cur = walk_below(cur, nxt, axis, T)
        pts.append(cur)
    chain = np.stack(pts, axis=1).reshape(-1, 3)
    lo = np.array(origin, np.float64)
    hi = lo.copy()
    hi[axis] += length
    if slab is not None:
        for k, d in enumerate(other):
            hi[d] += slab[k]
    return Case(np.concatenate([lo[None], chain, hi[None]]).astype(f32), tol, chains=(n_chains, beads), slab=slab is not None, seed=seed)


def straddle_case(length, tol, axis, origin, count=64, seed=0):
    """Pairs that the former fp32 cell formula (prefix_grid, a restatement) puts two cells apart although their fp32 d2 is
    below T, found by search among near-tolerance pairs on a line from `origin` over `length` metres."""
    rng = np.random.default_rng(seed)
    T = t2_of(tol)
    lo = np.array(origin, f32)
    hi = lo.copy()
    hi[axis] = f32(float(lo[axis]) + length)
    anchors = np.stack([lo, hi])
    _, g_lo, inv, dims = prefix_grid(anchors, tol)
    picked = []
    for _ in range(8):
        a = np.broadcast_to(lo, (1 << 21, 3)).copy()
        a[:, axis] = (float(lo[axis]) + rng.uniform(2 * tol, length - 3 * tol, len(a))).astype(f32)
        b = a.copy()
        b[:, axis] = (a[:, axis] + f32(tol)).astype(f32)
        b = walk_below(a, b, axis, T)
        ca = np.floor(((a[:, axis] - g_lo[axis]).astype(f32) * inv).astype(f32))
        cb = np.floor(((b[:, axis] - g_lo[axis]).astype(f32) * inv).astype(f32))
        hit = np.flatnonzero(cb - ca > 1)
        picked += [(a[i], b[i]) for i in hit]
        if len(picked) >= 4 * count:
            break
    picked.sort(key=lambda p: float(p[0][axis]))
    kept, last = [], -np.inf
    for a, b in picked:                  # pairs at least 1 m apart: each pair is its own cluster
        if float(a[axis]) - last > 1.0:
            kept += [a, b]
            last = float(b[axis])
        if len(kept) >= 2 * count:
            break
    return Case(np.concatenate([anchors[:1], np.array(kept, f32), anchors[1:]]), tol, straddling=len(kept) // 2)


WITNESS = np.array([0xC0E9EB88, 0x42855AD4, 0x42856511], dtype=np.uint32).view(f32)


def witness_case():
    xyz = np.zeros((3, 3), f32)
    xyz[:, 0] = WITNESS
    return Case(xyz, 0.02)


def blobs(rng, centres, side, per_blob):
    """Dense random blobs: `per_blob` points uniform in a cube of edge `side` around each centre."""
    return np.concatenate([c + rng.uniform(-side / 2, side / 2, (per_blob, 3)) for c in centres])


def cube_case(edge, tol, blob_side, n_blobs=12, per_blob=400, clutter=300, dup=50, seed=0):
    """A cloud spanning `edge` on every axis from an unround corner: blobs of edge `blob_side` (connected at `tol`),
    exact duplicates of some points, and random clutter."""
    rng = np.random.default_rng(seed)
    lo = np.array([-0.3170013, 0.2190007, 0.8130011]) * min(edge, 1.0)
    cen = lo + rng.uniform(0.1, 0.9, (n_blobs, 3)) * edge
    parts = [lo[None], (lo + edge)[None], blobs(rng, cen, blob_side, per_blob), lo + rng.uniform(0, edge, (clutter, 3))]
    xyz = np.concatenate(parts).astype(f32)
    xyz = np.concatenate([xyz, xyz[rng.integers(0, len(xyz), dup)]])
    return Case(xyz[rng.permutation(len(xyz))], tol, mn=1, seed=seed)


def micro_case(tol, seed=0):
    """A 1 m cube whose clusters live near the origin, where fp32 spacing is far finer than `tol`: blobs of edge 4 tol
    at a few tol from 0, duplicates, and clutter over the whole cube."""
    rng = np.random.default_rng(seed)
    cen = rng.uniform(2, 40, (6, 3)) * tol
    xyz = np.concatenate([[[0.0, 0.0, 0.0], [1.0, 1.0, 1.0]], blobs(rng, cen, 4 * tol, 200), rng.uniform(0, 1, (500, 3))]).astype(f32)
    xyz = np.concatenate([xyz, xyz[rng.integers(0, len(xyz), 100)]])
    return Case(xyz[rng.permutation(len(xyz))], tol)


def far_case(r, seed=0):
    """Points at +-r on every axis (the eight corners, some twice, and r with its fp32 successor) around an ordinary
    blob scene at the origin, tolerance 0.02."""
    rng = np.random.default_rng(seed)
    corners = np.array([[sx, sy, sz] for sx in (-r, r) for sy in (-r, r) for sz in (-r, r)], np.float64)
    rr = np.float64(np.nextafter(f32(r), f32(np.inf)))
    extra = np.array([[r, 0, 0], [rr, 0, 0], [0, -r, 0], [0, -r, 0], [0, 0, r], [0, 0, rr]])
    scene = blobs(rng, rng.uniform(-0.6, 0.6, (5, 3)), 0.08, 300)
    xyz = np.concatenate([corners, corners[:3], extra, scene]).astype(f32)
    return Case(xyz[rng.permutation(len(xyz))], 0.02)


def two_singletons_case():
    rng = np.random.default_rng(5)
    xyz = np.full((1000, 3), np.nan, f32)
    xyz[rng.random(1000) < 0.3] = np.inf
    xyz[rng.random(1000) < 0.2, 2] = -np.inf
    xyz[rng.random(1000) < 0.2, 1] = 0.5           # finite y and z, non-finite x
    xyz[137] = (-12345.678, 0.25, 1.5)
    xyz[861] = (54321.5, -3.0, 2.0)
    return Case(xyz, 0.02)


def nonfinite_case(seed=3):
    """A blob scene with NaN, +inf or -inf in one coordinate of 15 % of the points."""
    rng = np.random.default_rng(seed)
    xyz = np.concatenate([blobs(rng, rng.uniform(-0.6, 0.6, (8, 3)) + [0, 0, 1.2], 0.1, 500), rng.uniform(-1, 1, (1000, 3)) + [0, 0, 1.2]]).astype(f32)
    xyz = xyz[rng.permutation(len(xyz))]
    bad = np.flatnonzero(rng.random(len(xyz)) < 0.15)
    xyz[bad, rng.integers(0, 3, len(bad))] = rng.choice(np.array([np.nan, np.inf, -np.inf], f32), len(bad))
    return Case(xyz, 0.02, mn=20)


def line(n, spacing, start=(0.0, 0.0, 0.0), axis=0):
    xyz = np.tile(np.array(start, np.float64), (n, 1))
    xyz[:, axis] += spacing * np.arange(n)
    return xyz


def reversed_chain_case(n=50_000):
    """One chain whose point indices run against its geometry: every union hooks to a root far below."""
    return Case(line(n, 0.014, (-3.21, 0.37, 1.1))[::-1], 0.02, chain_sizes=[n])


def strided_chain_case(n=50_021, stride=7919):
    """One chain whose k-th bead is point (k * stride) mod n: neighbours along the chain are far apart in index."""
    geo = line(n, 0.014, (-3.21, 0.37, 1.1))
    xyz = np.empty_like(geo)
    xyz[(np.arange(n) * stride) % n] = geo
    return Case(xyz, 0.02, chain_sizes=[n])


def zipped_chains_case(n=30_000):
    """Two chains, one along x and one along y, with interleaved indices (even: the first, odd: the second) that meet only
    at their far ends."""
    a = line(n, 0.015, (0.0, 0.0, 1.0), 0)
    b = line(n, 0.015, (a[-1, 0] + 0.01, -(n - 1) * 0.015, 1.0), 1)   # its last bead lies 1 cm from the first chain's last
    xyz = np.empty((2 * n, 3))
    xyz[0::2], xyz[1::2] = a, b
    return Case(xyz, 0.02, chain_sizes=[2 * n])


def sphere_case(n=100_000, seed=11):
    """A Fibonacci sphere of n points about 1.2 cm apart, in random index order: one component."""
    k = np.arange(n) + 0.5
    phi = np.arccos(1 - 2 * k / n)
    theta = np.pi * (1 + 5 ** 0.5) * k
    r = 1.07
    xyz = np.stack([r * np.cos(theta) * np.sin(phi), r * np.sin(theta) * np.sin(phi), 2.0 + r * np.cos(phi)], axis=1)
    return Case(xyz[np.random.default_rng(seed).permutation(n)], 0.02, chain_sizes=[n])


def copies_case(n=10_000):
    """n copies of one point (d2 = 0) among a few others."""
    xyz = np.concatenate([np.tile([[0.4321, -0.1234, 1.5678]], (n, 1)), [[0.4321, -0.1234, 1.6], [3.0, 3.0, 3.0]]])
    return Case(xyz[np.random.default_rng(1).permutation(len(xyz))], 0.02, chain_sizes=[n, 1, 1])


def sheet_case(side=450, seed=2):
    """A wavy sheet of side^2 (about 200 k) points, 1.2 cm apart with jitter, in random index order: one component."""
    rng = np.random.default_rng(seed)
    u, v = np.meshgrid(np.arange(side) * 0.012, np.arange(side) * 0.012, indexing="ij")
    xyz = np.stack([u, v, 1.5 + 0.05 * np.sin(3 * u) * np.cos(2 * v)], axis=-1).reshape(-1, 3) - [2.7, 2.7, 0]
    xyz += rng.uniform(-0.0008, 0.0008, xyz.shape)
    return Case(xyz[rng.permutation(len(xyz))], 0.02, chain_sizes=[side * side])


def sized_clusters(sizes, seed, spacing=0.5):
    """Compact clusters of the given sizes (the first s points, in lexicographic order, of a 1 cm lattice cube) on a
    40 x 40 x n grid of `spacing`, indices shuffled."""
    rng = np.random.default_rng(seed)
    parts = []
    for k, s in enumerate(sizes):
        c = np.array([(k % 40) * spacing, (k // 40 % 40) * spacing, 1.0 + (k // 1600) * spacing])
        m = int(np.ceil(s ** (1 / 3) - 1e-9))
        cube = np.stack(np.meshgrid(np.arange(m), np.arange(m), np.arange(m), indexing="ij"), -1).reshape(-1, 3)[:s]
        parts.append(c + 0.01 * cube)
    xyz = np.concatenate(parts)
    return xyz[rng.permutation(len(xyz))]


def limits_case(mn, mx):
    sizes = [9, 10, 11, 19, 20, 21] * 5
    return Case(sized_clusters(sizes, 4), 0.02, mn=mn, mx=mx, chain_sizes=sorted(sizes, reverse=True))


def ties_case():
    """60 clusters of 7 points and 10 of 8, interleaved in index order: ranks among equal sizes follow the lowest index."""
    sizes = [7] * 60 + [8] * 10
    return Case(sized_clusters(sizes, 6), 0.02, mn=2, chain_sizes=sorted(sizes, reverse=True))


def singletons_case(n=3000):
    g = np.stack(np.meshgrid(np.arange(15), np.arange(15), np.arange(14), indexing="ij"), -1).reshape(-1, 3)[:n] * 0.05
    return Case(g[np.random.default_rng(8).permutation(n)], 0.02, chain_sizes=[1] * n)


def many_clusters_case(n_pass):
    """n_pass clusters of 2-5 points that pass min_size 2, plus 300 singletons that do not."""
    rng = np.random.default_rng(n_pass)
    sizes = list(rng.integers(2, 6, n_pass)) + [1] * 300
    return Case(sized_clusters(sizes, 9, spacing=0.1), 0.02, mn=2, chain_sizes=sorted([s for s in sizes if s >= 2], reverse=True))


def tiles_case():
    """A 12 000-point cluster whose points are spread over 30 000 indices: cluster_cloud scans 8 tiles of 4096."""
    sizes = [12_000] + [150] * 120
    return Case(sized_clusters(sizes, 10), 0.02, mn=100, chain_sizes=sorted(sizes, reverse=True))


def kinect_case():
    """The model builder's input: a synthetic Kinect frame of 8 objects, the table cut away, downsampled at a 1 cm leaf."""
    objs = synth.default_objects(8, seed=3)
    pts, oid = synth.render(0, objs)
    keep = (oid >= 0) & np.isfinite(pts["x"])
    ds = oracle.voxel_grid_exact(pts[keep], 0.01, 2, 0.0, 10.0)
    return Case(np.stack([ds["x"], ds["y"], ds["z"]], axis=1), 0.02, mn=50, mx=25000)


ORG = (-7.3100013, -0.4137021, -123.4567)
ORG2 = (-123.4567, -7.3100013, -7.3100013)
CASES = {
    **{"boundary-%g" % t: functools.partial(boundary_case, t) for t in (0.02, 0.005, 0.05, 0.007, 0.0123)},
    "witness": witness_case,
    "chain-80m-x-0.02": functools.partial(chains_case, 80.0, 0.02, 0, ORG),
    "chain-80m-x-0.005": functools.partial(chains_case, 80.0, 0.005, 0, ORG2, seed=1),
    "chain-400m-y-0.02": functools.partial(chains_case, 400.0, 0.02, 1, ORG2, seed=2),
    "chain-400m-y-0.005": functools.partial(chains_case, 400.0, 0.005, 1, ORG, seed=3),
    "chain-2000m-z-0.02": functools.partial(chains_case, 2000.0, 0.02, 2, ORG, seed=4),
    "chain-2000m-z-0.005": functools.partial(chains_case, 2000.0, 0.005, 2, ORG2, seed=5),
    "slab-80m-x-0.02": functools.partial(chains_case, 80.0, 0.02, 0, ORG, slab=(2.0, 0.1), seed=6),
    "slab-400m-y-0.005": functools.partial(chains_case, 400.0, 0.005, 1, ORG2, slab=(0.05, 0.01), seed=7),
    "slab-2000m-x-0.02": functools.partial(chains_case, 2000.0, 0.02, 0, ORG, slab=(0.1, 0.1), seed=8),
    "straddle-80m-x-0.02": functools.partial(straddle_case, 80.0, 0.02, 0, ORG, seed=1),
    "straddle-400m-y-0.02": functools.partial(straddle_case, 400.0, 0.02, 1, ORG2, seed=2),
    "straddle-2000m-z-0.02": functools.partial(straddle_case, 2000.0, 0.02, 2, ORG, seed=3),
    "straddle-2000m-x-0.005": functools.partial(straddle_case, 2000.0, 0.005, 0, ORG2, seed=4),
    "cube-5m-0.02": functools.partial(cube_case, 5.0, 0.02, 0.08),
    "cube-1km-0.02": functools.partial(cube_case, 1000.0, 0.02, 0.08, seed=1),
    "cube-1m-1e-12": functools.partial(micro_case, 1e-12),
    "cube-1m-1e-15": functools.partial(micro_case, 1e-15, seed=1),
    "far-1e13": functools.partial(far_case, 1e13),
    "far-3e38": functools.partial(far_case, 3e38, seed=1),
    "two-finite-singletons": two_singletons_case,
    "nan-inf-mixed": nonfinite_case,
    "chain-reversed": reversed_chain_case,
    "chain-strided": strided_chain_case,
    "chains-zipped": zipped_chains_case,
    "sphere-100k-permuted": sphere_case,
    "copies-10k": copies_case,
    "sheet-200k": sheet_case,
    "sizes-10-20": functools.partial(limits_case, 10, 20),
    "sizes-11-11": functools.partial(limits_case, 11, 11),
    "ties": ties_case,
    "singletons": singletons_case,
    "clusters-4096": functools.partial(many_clusters_case, MAX_CLUSTERS),
    "clusters-4097": functools.partial(many_clusters_case, MAX_CLUSTERS + 1),
    "extract-tiles": tiles_case,
    "kinect-downsampled": kinect_case,
}
NAMES = list(CASES)


@functools.lru_cache(maxsize=None)
def case(name):
    return CASES[name]()


@functools.lru_cache(maxsize=None)
def ref(name):
    c = case(name)
    return reference(c.xyz, c.tol, c.mn, c.mx)


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32).reshape(len(a), 4)


# ------------------------------------------------------------------ CPU: the oracle and the cases
@pytest.mark.parametrize("name", NAMES)
def test_oracle_equals_reference(name):
    c = case(name)
    labels, sizes, _ = ref(name)
    got_labels, got_sizes = oracle.euclidean_clusters(c.pts, c.tol, c.mn, c.mx)
    assert got_sizes.tolist() == sizes.tolist()
    assert np.array_equal(got_labels, labels)


@pytest.mark.parametrize("name", NAMES)
def test_grid_keeps_every_joined_pair_adjacent(name):
    """The grid sizing and cell formula of pft_cluster.cu, restated in fp64: at most 2^22 cells, and every pair the
    reference joins lies in neighbouring cells, so a 27-cell neighbourhood compares it."""
    c = case(name)
    _, _, edges = ref(name)
    cells, dims = fixed_cells(c.xyz, c.tol)
    assert int(np.prod(dims)) <= MAX_CELLS and dims.max() <= MAX_CELLS
    assert len(straddles(cells, edges)) == 0


@pytest.mark.parametrize("tol", [0.02, 0.005, 0.05, 0.007, 0.0123])
def test_boundary_case_reaches_every_target(tol):
    c = case("boundary-%g" % tol)
    assert set(c.props["boundary_targets"]) <= c.props["found"]
    labels, sizes, _ = ref("boundary-%g" % tol)
    d2 = d2_f32(c.xyz[0::2], c.xyz[1::2])
    joined = labels[0::2] == labels[1::2]
    assert np.array_equal(joined, d2 < t2_of(tol)) and joined.any() and (~joined).any()


def test_boundary_tolerances_include_both_roundings():
    same = [t2_of(t) == f32(t) * f32(t) for t in (0.02, 0.005, 0.05, 0.007, 0.0123)]
    assert any(same) and not all(same)
    assert f32(0.0123 * 0.0123) > f32(0.0123) * f32(0.0123) and f32(0.05 * 0.05) < f32(0.05) * f32(0.05)


@pytest.mark.parametrize("name", ["witness"] + [n for n in NAMES if n.startswith("straddle-")])
def test_former_grid_misses_joined_pairs(name):
    """The former fp32 cell formula puts pairs that the reference joins two cells apart: a GPU built on it splits them."""
    c = case(name)
    labels, _, edges = ref(name)
    missed = straddles(prefix_cells(c.xyz, c.tol), edges)
    if name == "witness":
        assert edges.tolist() == [[1, 2]] and missed.tolist() == [0]
        assert prefix_cells(c.xyz, c.tol)[:, 0].tolist() == [0, 3698, 3700]
    else:
        assert len(missed) == c.props["straddling"] >= 8


@pytest.mark.parametrize("name", [n for n in NAMES if n.startswith(("chain-", "slab-")) and "m-" in n])
def test_chains_are_the_clusters(name):
    c = case(name)
    n_chains, beads = c.props["chains"]
    _, sizes, _ = ref(name)
    assert sizes.tolist() == [beads] * n_chains + [1, 1]
    it, _, _, dims = prefix_grid(c.xyz, c.tol)
    assert it == 0                                        # the narrow cell: no doubling
    assert max(dims) >= 4000 and (sorted(dims)[1] > 1) == c.props["slab"]


@pytest.mark.parametrize("name,doublings", [("cube-5m-0.02", 1), ("cube-1km-0.02", 9), ("cube-1m-1e-12", 33)])
def test_cell_size_cases_double_the_former_cell(name, doublings):
    c = case(name)
    assert prefix_grid(c.xyz, c.tol)[0] == doublings
    _, sizes, _ = ref(name)
    assert (sizes > 100).sum() >= 6                       # the blobs are clusters


@pytest.mark.parametrize("name", ["cube-1m-1e-15", "far-1e13", "far-3e38"])
def test_extreme_cases_overrun_the_former_sizing_loop(name):
    c = case(name)
    assert prefix_grid(c.xyz, c.tol)[0] is None


def test_extreme_cases_have_their_shape():
    _, sizes, _ = ref("two-finite-singletons")
    assert sizes.tolist() == [1, 1] and np.isfinite(case("two-finite-singletons").xyz).all(axis=1).sum() == 2
    c = case("nan-inf-mixed")
    for v in (np.nan, np.inf, -np.inf):
        for d in range(3):
            assert (np.isnan(c.xyz[:, d]) if np.isnan(v) else c.xyz[:, d] == v).any()
    for name, r in (("far-1e13", 1e13), ("far-3e38", 3e38)):
        labels, sizes, _ = ref(name)
        far = np.abs(case(name).xyz).max(axis=1) >= f32(r)
        assert far.sum() == 17 and len(set(labels[far].tolist())) < 17   # duplicated corners join, distinct ones do not
    _, sizes, _ = ref("cube-1m-1e-15")
    assert (sizes >= 100).sum() == 6


@pytest.mark.parametrize("name", ["chain-reversed", "chain-strided", "chains-zipped", "sphere-100k-permuted", "copies-10k", "sheet-200k",
                                  "sizes-10-20", "sizes-11-11", "ties", "singletons", "clusters-4096", "clusters-4097", "extract-tiles"])
def test_built_components(name):
    c = case(name)
    _, sizes, _ = ref(name)
    want = [s for s in c.props["chain_sizes"] if c.mn <= s <= c.mx]
    assert sizes.tolist() == want
    if name == "sizes-11-11":
        assert want == [11] * 5
    if name.startswith("clusters-"):
        assert len(want) == int(name.split("-")[1])


def test_tie_ranks_follow_the_lowest_index():
    labels, sizes, _ = ref("ties")
    low = [int(np.flatnonzero(labels == k)[0]) for k in range(len(sizes))]
    assert sizes.tolist() == [8] * 10 + [7] * 60
    assert low[:10] == sorted(low[:10]) and low[10:] == sorted(low[10:]) and low != sorted(low)


def test_reference_on_a_known_answer():
    """Two chains 1.5 cm apart in bead spacing, 5 cm between them, and a point exactly at the tolerance of a chain end."""
    a = line(30, 0.015, (0, 0, 1))
    b = line(20, 0.015, (0, 0.05, 1))
    end = a[-1] + [0, 0, 0]
    p = np.array([[end[0] + 0.02, 0, 1]])       # (float)0.02 from the end: d2 == (float)(0.02^2) is not joined
    xyz = np.concatenate([a, b, p]).astype(f32)
    labels, sizes, edges = reference(xyz, 0.02, 1, BIG)
    joined = d2_f32(xyz[29], xyz[50]) < t2_of(0.02)
    assert sizes.tolist() == ([31, 20] if joined else [30, 20, 1])
    assert (labels[:30] == 0).all() and (labels[30:50] == 1).all() and len(edges) == 29 + 19 + int(joined)


# ------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("name", NAMES)
def test_gpu_clusters_equal_reference(name):
    c = case(name)
    labels, sizes, _ = ref(name)
    cloud = pcl.PointCloud(c.pts)
    ec = pcl.EuclideanClusterExtraction()
    ec.setClusterTolerance(c.tol); ec.setMinClusterSize(c.mn); ec.setMaxClusterSize(c.mx); ec.setInputCloud(cloud)
    if len(sizes) > MAX_CLUSTERS:
        with pytest.raises(pcl.capi.PftError) as e:
            ec.extract()
        assert e.value.code == pcl.capi.ERR_CAPACITY
        return
    clusters = ec.extract()
    assert ec.sizes.tolist() == sizes.tolist()
    assert np.array_equal(ec.labels, labels)
    out = pcl.PointCloud()
    for k, idx in enumerate(clusters):
        got = ec.cluster_cloud(k, out).to_numpy()
        assert np.array_equal(_bits(got), _bits(c.pts[idx])), k
    first = ec.labels.copy()
    ec.extract()                                          # the lock-free union-find is deterministic
    assert np.array_equal(ec.labels, first)
