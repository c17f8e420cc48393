"""The O(N) particle stages against exact references, at every launch shape up to 100 000 particles.

normalize_kernel, update_kernel, cdf_kernel, resample_kernel / alias_table_kernel and kld_insert_kernel /
kld_stop_kernel decide which particles survive and which pose is published.  Above a capacity of 4096 the first three
run as one cluster of 8 CTAs (launch_replicated) whose per-CTA partials travel through distributed shared memory.
Every stage here is O(N), so numpy and the CPU oracle restate it exactly in milliseconds even at 100 000 particles, and
the comparisons can be bit for bit:

  normalise   numpy float64 restatement of normalizeWeight, the weight sum exact (math.fsum) and then rounded
  update      exact sums of the fp32 terms (double)(float)(s * w), rounded once
  resample    the oracle with injected draws; its build_cdf / sample_cdf restate the 2^-40 fixed-point table
  KLD         the oracle, and a numpy restatement of the bin keys, the stop rule and the hash of kld_insert_kernel

A float64 value whose float32 rounding could change under the error of the GPU's own arithmetic (CUDA's double exp is
not correctly rounded; the fp64 tree sums have rounding error) is flagged: flagged entries may differ by one float32
ulp, all others must be bit-identical.  Where the inputs are constructed, a CPU test asserts nothing is flagged, so the
GPU test requires bit equality outright.

Shapes: the single-CTA capacities up to 4096, the cluster capacities above it (8191-8193 straddle the 8 x 1024 thread
stride, 100 003 is odd), and a tracker that once held 100 000 particles and now holds a few: capacity only grows, so
the cluster kernels run on 1-150 live particles with a stale tail behind them.

The tests without the gpu mark check on the CPU that every constructed case has the property it targets (boundary
draws on exact table entries, extremes in CTA 7 of the cluster, keys sharing one home slot, stops at the scan tile
edges) and that the numpy references agree with the oracle."""
import functools
import math

import numpy as np
import pytest

import oracle
from pcl_tracking_b200 import pcl
from tests import util

f32 = np.float32
STATE = ("x", "y", "z", "roll", "pitch", "yaw")
DBL_MAX = float(np.finfo(np.float64).max)
FILL = f32(-3.4e38)                 # raw slots past the live count: any read of one moves the minimum
TWO40 = 2.0 ** 40                   # the cumulative table's fixed point
CLUSTER_CTAS, CTA_THREADS = 8, 1024  # kClusterCtas x the replicated kernels' block size
MOTION_RATIO = f32(0.25)
ALPHAS = (15.0, 1.0, 200.0)
BIN = f32(0.05)

SINGLE_CAPS = (1, 2, 3, 31, 1024, 4095, 4096)
CLUSTER_CAPS = (4097, 8191, 8192, 8193, 65537, 100000, 100003)
STALE_CAP, STALE_LIVE = 100000, (1, 2, 3, 7, 9, 150)
SHAPES = [(c, None) for c in SINGLE_CAPS + CLUSTER_CAPS] + [(STALE_CAP, n) for n in STALE_LIVE]
NORM_SHAPES = ([(c, n, 2) for c, n in SHAPES] + [(c, None, 3) for c in (31, 4097, 8191, 100000)]
               + [(c, None, 8) for c in (31, 4095, 8193, 65537, 100003)])
KLD_NMAX = (4097, 20000, 100000)
STOP_AT = (4095, 4096, 4097, 70001)  # around the 4096-entry tiles of block_exclusive_scan, and one far out


def shape_id(v):
    return "-".join("x" if x is None else str(x) for x in v) if isinstance(v, tuple) else str(v)


# ------------------------------------------------------------------ float32 rounding under a bounded error
def f32_ambiguous(x64, err):
    """True where the float32 rounding of x64 could change under an error of `err`: x64 lies within err of a float32
    rounding midpoint."""
    x = np.asarray(x64, np.float64)
    with np.errstate(over="ignore", invalid="ignore"):
        f = x.astype(f32)
        fd = f.astype(np.float64)
        lo = (fd + np.nextafter(f, f32(-np.inf)).astype(np.float64)) / 2
        hi = (fd + np.nextafter(f, f32(np.inf)).astype(np.float64)) / 2
        return (np.abs(x - lo) <= err) | (np.abs(x - hi) <= err)


def fp64_sum_error(terms):
    """A bound on the error of an fp64 sum of the float32 `terms` in any order: 0 when every partial sum is exact (all
    terms are multiples of a power of two g and sum |t| < 2^53 g), else (n - 1) 2^-53 sum |t|."""
    t = np.abs(np.asarray(terms, np.float64))
    t = t[t != 0]
    if len(t) < 2:
        return 0.0
    mant, e = np.frexp(t)
    m = (mant * 2.0 ** 24).astype(np.int64)  # a float32's significand: an integer
    g = float(np.min(np.ldexp((m & -m).astype(np.float64), e - 24)))
    a = math.fsum(t.tolist())
    return 0.0 if a < 2.0 ** 53 * g else (len(t) - 1) * 2.0 ** -53 * a * 1.001


def within_one_ulp(a, b):
    a, b = np.asarray(a, f32), np.asarray(b, f32)
    return (a.view(np.uint32) == b.view(np.uint32)) | (a == np.nextafter(b, f32(np.inf))) | (a == np.nextafter(b, f32(-np.inf)))


def assert_flagged_equal(got, want, flag, what):
    """Unflagged entries bit-identical, flagged ones within one float32 ulp."""
    got, want = np.atleast_1d(np.asarray(got, f32)), np.atleast_1d(np.asarray(want, f32))
    flag = np.broadcast_to(np.asarray(flag, bool), got.shape)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    bad = (got.view(np.uint32) != want.view(np.uint32)) & (~flag | ~within_one_ulp(got, want))
    if bad.any():
        i = np.flatnonzero(bad)[:5]
        raise AssertionError(f"{what}: {int(bad.sum())} of {got.size} differ, at {i.tolist()}: got {got[i].tolist()} want {want[i].tolist()}")


# ------------------------------------------------------------------ references
def ref_normalize(raw, alpha):
    """normalize_kernel in float64: (weights, flagged, w_min).  w_min over all weights, w_max over the non-zero ones;
    equal: 1/n each; else (float)exp(1 - alpha (w - w_min) / (w_max - w_min)) per non-zero weight, each divided by the
    float32 of the weight sum."""
    w = np.asarray(raw, f32).astype(np.float64)
    n = len(w)
    wmin = float(w.min())
    nz = w[w != 0]
    wmax = float(nz.max()) if len(nz) else -DBL_MAX
    flag = np.zeros(n, bool)
    if wmax != wmin:
        with np.errstate(over="ignore", under="ignore"):
            e = np.exp(1.0 - alpha * (w - wmin) / (wmax - wmin))
            v = np.where(w != 0, e.astype(f32), f32(0))
        flag = (w != 0) & f32_ambiguous(e, 4 * np.spacing(e))  # CUDA's double exp: within 1-2 fp64 ulps
    else:
        v = np.full(n, f32(1) / f32(n), f32)
    s = math.fsum(v.astype(np.float64).tolist())
    if s != 0.0:
        err = fp64_sum_error(v)
        if err > 0 and f32_ambiguous(s, err):  # (an exact sum rounds as the reference does, midpoint or not)
            flag[:] = True
        out = v / f32(s)
    else:
        out = np.full(n, f32(1) / f32(n), f32)
    return out.astype(f32), flag, wmin


def ref_update(parts, rep_old):
    """update(): (rep, motion, flags per state field).  rep = the exact sum of the terms (float)((double)s * (double)w)
    rounded once; motion = rep - rep_old in float32; rep.weight = 1.0f / n."""
    n = len(parts)
    w = parts["weight"].astype(np.float64)
    rep = np.zeros(1, pcl.PARTICLE)[0]
    mot = np.zeros(1, pcl.PARTICLE)[0]
    flags = {}
    for k in STATE:
        terms = (parts[k].astype(np.float64) * w).astype(f32).astype(np.float64)
        s = math.fsum(terms.tolist())
        rep[k] = f32(s)
        err = fp64_sum_error(terms)
        flags[k] = bool(err > 0 and f32_ambiguous(s, err))
        mot[k] = f32(rep[k]) - f32(rep_old[k])
    rep["one"], rep["weight"] = f32(1), f32(1) / f32(n)
    mot["one"], mot["weight"] = f32(1), f32(0)
    return rep, mot, flags


def assert_pose_equal(got, want, flags, what):
    for k in ("one", "weight") + STATE:
        assert_flagged_equal(got[k], want[k], flags.get(k, False), f"{what}.{k}")


def build_cdf(w):
    """The 2^-40 fixed-point cumulative table (cdf_kernel, the oracle's build_cdf): each weight truncated."""
    w = np.asarray(w, f32).astype(np.float64)
    q = np.where(w > 0, np.floor(w * TWO40), 0).astype(np.uint64)
    return np.cumsum(q, dtype=np.uint64)


def sample_cdf(cdf, u):
    """cdf_pick: the first j with cdf[j] > (uint64)(u * total); total 0: (int)(u * n)."""
    n, total = len(cdf), int(cdf[-1])
    u = np.asarray(u, np.float64)
    if total == 0:
        return np.minimum((u * n).astype(np.int64), n - 1)
    t = (u * float(total)).astype(np.uint64)
    return np.minimum(np.searchsorted(cdf, t, side="right"), n - 1)


def kld_hash(keys):
    """kld_insert_kernel's hash of a 6-int bin key (FNV-1a steps, each followed by h ^= h >> 15)."""
    h = np.full(len(keys), 2166136261, dtype=np.uint64)
    for d in range(6):
        h = ((h ^ (np.asarray(keys)[:, d].astype(np.int64) & 0xFFFFFFFF).astype(np.uint64)) * np.uint64(16777619)) & np.uint64(0xFFFFFFFF)
        h ^= h >> np.uint64(15)
    return h


def kld_table_size(cap):
    ts = 1024
    while ts < 2 * cap:
        ts <<= 1
    return ts


def bin_keys(states):
    """(int)(x / bin_size) per component: float32 division, truncation toward zero."""
    return np.trunc(np.asarray(states, f32) / BIN).astype(np.int64)


@functools.lru_cache(maxsize=None)
def kl_table(n, delta, eps):
    return np.array([0.0, 0.0] + [oracle.kl_bound(k, delta, eps) for k in range(2, n + 2)])


def kld_count(keys, delta=0.99, eps=0.2):
    """The first n >= 1 with !(n < n_max && (k(n) < 2 || n < KLbound(k(n)))), k(n) = distinct keys among the first n."""
    n_max = len(keys)
    _, first = np.unique(np.asarray(keys), axis=0, return_index=True)
    new = np.zeros(n_max, bool)
    new[first] = True
    k = np.cumsum(new)
    n = np.arange(1, n_max + 1)
    go_on = (n < n_max) & ((k < 2) | (n < kl_table(n_max, delta, eps)[k]))
    return int(n[~go_on][0])


# ------------------------------------------------------------------ inputs
def particles(n, seed=1):
    return util.particles_around(np.array([0.11, -0.07, 1.23]), n, seed=seed)


def extreme_positions(n):
    """name -> (index of the global minimum, index of the global maximum).  Particle i of the normalise is read by CTA
    (i / 1024) % 8 of the cluster; CTA 7 owns the indices in [7168 + 8192 k, 8192 + 8192 k)."""
    out = {"cta0": (0, min(1023, n - 1)), "tile": (min(1023, n - 1), min(1024, n - 1)),
           "stride": (min(8191, n - 1), min(8192, n - 1)), "last": (n - 1, 0)}
    cta7 = np.flatnonzero((np.arange(n) // CTA_THREADS) % CLUSTER_CTAS == CLUSTER_CTAS - 1)
    if len(cta7) > 1:
        out["cta7"] = (int(cta7[-1]), int(cta7[0]))
    return {k: v for k, v in out.items() if v[0] != v[1]}


def raw_patterns(n, seed):
    """name -> raw weights (float32, n)."""
    rng = np.random.default_rng(seed)
    real = (-rng.uniform(20, 300, n)).astype(f32)  # raw weight = -(sum of the coherences of ~300 model points)
    out = {"realistic": real}
    z = real.copy()
    z[rng.random(n) < 0.1] = 0
    out["zeros10"] = z
    out["all_zero"] = np.zeros(n, f32)
    out["all_equal"] = np.full(n, f32(-123.5))
    u = np.where(rng.random(n) < 0.5, f32(-7.25), f32(0)).astype(f32)
    u[0] = f32(-7.25)
    out["one_value_and_zeros"] = u
    v = f32(-50.0)
    out["one_ulp"] = np.where(np.arange(n) % 3 == 1, np.nextafter(v, f32(0)), v).astype(f32)
    span = -(10.0 ** rng.uniform(-38, math.log10(3e38), n))
    span[0], span[-1] = -3e38, -1e-38
    out["span"] = span.astype(f32)
    for name, (imin, imax) in extreme_positions(n).items():
        r = real.copy()
        r[imin], r[imax] = f32(-1000), f32(-1)
        out["extremes_" + name] = r
    return out


def raw_slices(raw, R, cap):
    """The gathered raw buffer [R][slice_cap]: particle i at raw_slot(i) = (i % R, i / R), FILL past the live count."""
    sc = -(-cap // R)
    s = np.full((R, sc), FILL, f32)
    i = np.arange(len(raw))
    s[i % R, i // R] = raw
    return s


def update_cases(n, seed):
    """Update inputs whose terms s * w are exact in float32 and whose fp64 sums are exact in any order: positions on a
    2^-10 m grid (2^-8 m at 100 m), angles on a 2^-10 rad grid plus exactly +-pi, weights m 2^-24 with m < 256 (powers
    of two where a state is +-pi or the weight dominates)."""
    rng = np.random.default_rng(seed)

    def mk(centre, step, m):
        p = particles(n, seed + 1)
        for k, c in zip(("x", "y", "z"), centre):
            p[k] = ((round(c / step) + rng.integers(-2000, 2001, n)) * step).astype(f32)
        for k in ("roll", "pitch", "yaw"):
            p[k] = (rng.integers(-3217, 3218, n) * 2.0 ** -10).astype(f32)
        p["roll"][0], p["pitch"][-1] = f32(np.pi), -f32(np.pi)
        m = m.copy()
        m[0], m[-1] = 64, 128
        p["weight"] = (m * 2.0 ** -24).astype(f32)
        return p

    m = rng.integers(0, 256, n)
    dom = np.ones(n, np.int64)
    dom[min(rng.integers(1, max(n - 1, 2)), n - 1)] = 1 << 23  # weight 1/2
    zeros = np.where(rng.random(n) < 0.5, 0, m)
    return {"near": mk((0.11, -0.07, 1.23), 2.0 ** -10, m), "far": mk((100.0, -100.0, 100.0), 2.0 ** -8, m),
            "dominant": mk((0.11, -0.07, 1.23), 2.0 ** -10, dom), "zeros": mk((1.2, 1.2, 1.2), 2.0 ** -10, zeros)}


def segment_edges(n):
    seg = ((-(-n // CLUSTER_CTAS)) + 3) & ~3
    return sorted({i for r in range(CLUSTER_CTAS) if r * seg < n for i in (r * seg, min(r * seg + seg, n) - 1)})


def split_units(k, rng, units=1 << 20):
    """k non-negative integers summing to `units`."""
    p = rng.random(k) ** 3 + 1e-3
    c = np.floor(p / p.sum() * units).astype(np.int64)
    c[np.argmax(c)] += units - c.sum()
    return c


def cdf_weights(n, kind, rng):
    """Selection weights of a cumulative-table case (float32)."""
    if kind == "all_tiny":  # every weight quantises to 0: the total == 0 uniform branch
        return (rng.uniform(1.0, 1.99, n) * 2.0 ** -41).astype(f32)
    w = np.zeros(n)
    if kind == "exact":  # multiples of 2^-20 summing to 1, a fifth of them zero: the table is exact
        nz = np.flatnonzero(rng.random(n) >= 0.2) if n > 1 else np.arange(n)
        nz = nz if len(nz) else np.arange(n)
    elif kind == "segments":  # non-zero only at the first and last index of each 8-CTA scan segment
        nz = np.array(segment_edges(n))
    elif kind == "tiny_interleaved":  # weights below 2^-40 (never picked) between exact ones
        nz = np.arange(n)[1::2] if n > 1 else np.arange(n)
    w[nz] = split_units(len(nz), rng) * 2.0 ** -20
    w = w.astype(f32)
    if kind == "tiny_interleaved":
        tiny = np.setdiff1d(np.arange(n), nz)
        w[tiny] = (rng.uniform(1.0, 1.99, len(tiny)) * 2.0 ** -41).astype(f32)
    return w


CDF_KINDS = ("exact", "segments", "tiny_interleaved", "all_tiny")


def selection_draws(w, stride, rng):
    """Selection uniforms on table boundaries u = cdf[j] 2^-40 (exact in float32), with u = 0 and u = 1 - 2^-24 mixed in."""
    cdf = build_cdf(w)
    total = int(cdf[-1])
    if total == 1 << 40:
        b = cdf[cdf < total].astype(np.float64) * 2.0 ** -40
        u = rng.choice(b, stride) if len(b) else np.zeros(stride)
    else:
        u = rng.random(stride)
    u = u.astype(f32)
    u[rng.random(stride) < 0.125] = 0
    u[rng.random(stride) < 0.125] = f32(1 - 2.0 ** -24)
    return u


def motion_draws(stride, rng):
    """u_motion at motion_ratio, one ulp below it, and random."""
    u = rng.random(stride).astype(f32)
    u[0::3] = MOTION_RATIO
    u[1::3] = np.nextafter(MOTION_RATIO, f32(0))
    return u


def resample_draws(w, stride, seed):
    rng = np.random.default_rng(seed)
    usel = selection_draws(w, stride, rng)
    normals = rng.standard_normal((stride, 6), dtype=f32)
    return usel[None], normals[None], motion_draws(stride, rng)[None]


# ------------------------------------------------------------------ KLD cases (zero step noise, quat 0: candidate n is particle n)
def states_of_keys(keys):
    k = np.asarray(keys, np.float64)
    return ((k + np.where(k >= 0, 0.5, -0.5)) * float(BIN)).astype(f32)


@functools.lru_cache(maxsize=None)
def chain_keys(ts, want=2048):
    """`want` distinct keys homed at the table's last slot (the probe wraps to slot 0), in groups that differ only in
    the sixth component: sweeping that component under a fixed prefix finds ~2^20 / ts keys per prefix."""
    rng = np.random.default_rng(17)
    six = np.arange(-(1 << 19), 1 << 19, dtype=np.int64)
    found = []
    while sum(len(f) for f in found) < want:
        keys = np.empty((len(six), 6), np.int64)
        keys[:, :5] = rng.integers(-30, 31, 5)
        keys[:, 5] = six
        found.append(keys[(kld_hash(keys) & np.uint64(ts - 1)) == ts - 1])
    return np.concatenate(found)[:want]


def kld_case(n_max, name):
    """Candidate states (n_max, 6) float32 of a KLD case."""
    rng = np.random.default_rng(n_max + len(name))
    a, b = states_of_keys([[3, -2, 24, 1, 0, -1]])[0], states_of_keys([[3, -2, 24, 1, 0, -2]])[0]
    if name == "one_bin":
        return np.tile(a, (n_max, 1))
    if name == "distinct":
        i = np.arange(n_max)
        return states_of_keys(np.stack([i % 40 - 20, i // 40 % 40 - 20, i // 1600 - 20, i % 7, -(i % 3), i % 2], axis=1))
    if name.startswith("stop_"):  # one bin until candidate T-1 opens a second: k(T) = 2 >= ... stops at T
        t = int(name[5:])
        s = np.tile(a, (n_max, 1))
        s[t - 1] = b
        return s
    if name == "straddle_zero":  # (int) truncates toward zero: (-bin, bin) is one bin, both signed zeros included
        s = rng.uniform(-0.1, 0.1, (n_max, 6)).astype(f32)
        s[rng.random((n_max, 6)) < 0.05] = f32(0)
        s[rng.random((n_max, 6)) < 0.05] = f32(-0.0)
        s[rng.random((n_max, 6)) < 0.05] = np.nextafter(BIN, f32(0)) * rng.choice([-1, 1])
        return s.astype(f32)
    if name == "bin_edges":  # exactly k * bin and one ulp either side
        s = (rng.integers(-1, 2, (n_max, 6)) * BIN).astype(f32)
        nudge = rng.integers(-1, 2, (n_max, 6))
        s = np.where(nudge > 0, np.nextafter(s, f32(np.inf)), np.where(nudge < 0, np.nextafter(s, f32(-np.inf)), s))
        return s.astype(f32)
    if name == "hash_chain":  # ~2000 keys with one home slot (the last), in sixth-component groups, then repeats
        keys = chain_keys(kld_table_size(n_max))
        return states_of_keys(keys[np.arange(n_max) % len(keys)])
    raise KeyError(name)


def kld_names(n_max):
    names = ["one_bin", "distinct", "straddle_zero", "bin_edges"] + [f"stop_{t}" for t in STOP_AT if t < n_max]
    return names + (["hash_chain"] if n_max == KLD_NMAX[0] else [])


def kld_old_set(states):
    """The old particle set: the candidate states with equal weights; selection u_n = (n + 1/2) / n_max picks particle n."""
    n = len(states)
    p = oracle.make_particles(states, np.full(n, f32(1) / f32(n)))
    usel = ((np.arange(n) + 0.5) / n).astype(f32)
    return p, usel


KLD_CASES = [(n, name) for n in KLD_NMAX for name in kld_names(n)]


# ------------------------------------------------------------------ trackers
@functools.lru_cache(maxsize=None)
def small_scene():
    return util.small_case(31, n_scene=600, n_model=40)


def make_tracker(cap, live=None, R=1, kld=False, n_max=None, **kw):
    """(gpu tracker, oracle) with `cap` particles of capacity and `live` (default cap) live ones."""
    g, o = util.make_pair(kld=kld, particle_num=cap, max_particle_num=n_max or cap, use_hsv=False, iteration_num=1, **kw)
    if R > 1:
        g.setShard(R, 0)
    scene, model, _ = small_scene()
    g.setReferenceCloud(model)
    g.setInputCloud(pcl.PointCloud(scene))  # (the tracker keeps the cloud alive)
    g.setParticles(particles(cap))
    if live is not None:
        g.setParticles(particles(live))
    return g, o


# ================================================================== CPU tests
def test_f32_ambiguous_midpoints():
    one_up = 1.0 + 2.0 ** -24      # midpoint of 1 and its upper neighbour
    one_down = 1.0 - 2.0 ** -25    # midpoint of 1 and its lower neighbour (the ulp halves below a power of two)
    big = 16777217.0               # midpoint of 2^24 and 2^24 + 2
    for m in (one_up, one_down, big, -one_up, 3 * 2.0 ** -150):
        assert f32_ambiguous(m, 0.0)
        assert f32_ambiguous(np.nextafter(m, np.inf), 2 * abs(np.spacing(m)))
        assert not f32_ambiguous(m + 4 * abs(np.spacing(m)), 2 * abs(np.spacing(m)))
    assert not f32_ambiguous(one_up + 2.0 ** -40, 2.0 ** -41)
    assert f32_ambiguous(one_up + 2.0 ** -40, 2.0 ** -39)
    assert not f32_ambiguous(1.0, 2.0 ** -30)
    assert not f32_ambiguous(one_down - 2.0 ** -45, 2.0 ** -46)
    assert not f32_ambiguous(3.4e38, 1e20)  # next to the largest float: no overflow, no midpoint
    np.testing.assert_array_equal(f32_ambiguous(np.array([1.0, one_up, 2.5]), 0.0), [False, True, False])


@pytest.mark.parametrize("cap,live,R", NORM_SHAPES, ids=shape_id)
def test_normalize_cases_are_exact(cap, live, R):
    """Every normalise case: the reference is unflagged, the extremes sit where they were put, and the slices place
    particle i at raw_slot(i) with FILL everywhere else."""
    n = live or cap
    for name, raw in raw_patterns(n, cap + n + R).items():
        for alpha in ALPHAS:
            _, flag, wmin = ref_normalize(raw, alpha)
            assert not flag.any(), (name, alpha, int(flag.sum()))
        if name.startswith("extremes_"):
            imin, imax = extreme_positions(n)[name[9:]]
            assert raw.argmin() == imin and raw.argmax() == imax
            if name == "extremes_cta7":
                assert (imin // CTA_THREADS) % CLUSTER_CTAS == 7 and (imax // CTA_THREADS) % CLUSTER_CTAS == 7
        s = raw_slices(raw, R, cap)
        i = np.arange(n)
        assert np.array_equal(s[i % R, i // R], raw) and (s == FILL).sum() == s.size - n
    if n > 7168:
        assert "extremes_cta7" in raw_patterns(n, 0)


def test_normalize_reference_agrees_with_oracle():
    n = 100000
    for name, raw in raw_patterns(n, 5).items():
        for alpha in ALPHAS:
            o = oracle.Tracker(kld=False)
            o.set_d(oracle.ALPHA, alpha)
            p = particles(n)
            p["weight"] = raw
            o.set_particles(p)
            o.normalize()
            want, flag, wmin = ref_normalize(raw, alpha)
            assert_flagged_equal(o.get_particles()["weight"], want, flag, f"{name} alpha {alpha}")
            assert o.fit_ratio() == wmin


def test_update_reference_agrees_with_oracle():
    n = 100000
    for name, p in update_cases(n, 3).items():
        o = oracle.Tracker(kld=False)
        old = p[5].copy()
        o.set_particles(p)
        o.set_result(old)
        o.update()
        rep, mot, flags = ref_update(p, old)
        got = o.get_result()
        for k in STATE:  # the oracle sums in fp32, one particle after another
            terms = np.abs((p[k].astype(np.float64) * p["weight"].astype(np.float64)).astype(f32).astype(np.float64))
            assert abs(float(got[k]) - float(rep[k])) <= n * 2.0 ** -24 * terms.sum() + np.spacing(abs(rep[k])), (name, k)
        assert got["weight"] == rep["weight"]


@pytest.mark.parametrize("cap,live", SHAPES, ids=shape_id)
def test_update_cases_are_exact(cap, live):
    n = live or cap
    for name, p in update_cases(n, cap + n).items():
        _, _, flags = ref_update(p, p[0])
        assert not any(flags.values()), (name, flags)


@pytest.mark.parametrize("cap,live", SHAPES, ids=shape_id)
def test_cdf_cases_hit_boundaries(cap, live):
    """Boundary draws land exactly on table entries, weights below 2^-40 are never picked, the segment case has its
    weight on segment edges only, and the numpy table and pick agree with the oracle's resample."""
    n = live or cap
    rng = np.random.default_rng(n)
    for kind in CDF_KINDS:
        w = cdf_weights(n, kind, rng)
        cdf = build_cdf(w)
        usel = selection_draws(w, n, np.random.default_rng(n + 1))
        if kind == "all_tiny":
            assert cdf[-1] == 0
        else:
            assert int(cdf[-1]) == 1 << 40
            t = (usel.astype(np.float64) * float(cdf[-1])).astype(np.uint64)
            on = np.isin(t, cdf) | (usel == 0)
            assert on.mean() > 0.7 or n < 8, (kind, on.mean())
        pick = sample_cdf(cdf, usel)
        if kind == "tiny_interleaved" and n > 1:
            assert np.all(pick % 2 == 1)
        if kind == "segments":
            assert set(np.flatnonzero(w)) <= set(segment_edges(n))
        if kind != "all_tiny":
            assert np.all(w[pick] > 0) or n == 1
        o = oracle.Tracker(kld=False)
        o.set_i(oracle.PARTICLE_NUM, n)
        o.set_i(oracle.SAMPLER, oracle.SAMPLER_CDF)
        p = particles(n)
        p["weight"] = w
        o.set_particles(p)
        o.inject_draws(usel[None], np.zeros((1, n, 6), f32), np.ones((1, n), f32))
        o.resample(0)
        np.testing.assert_array_equal(o.ancestors()[1:], pick[1:], err_msg=kind)


@pytest.mark.parametrize("n_max,name", KLD_CASES, ids=shape_id)
def test_kld_cases_have_their_targets(n_max, name):
    states = kld_case(n_max, name)
    keys = bin_keys(states)
    p, usel = kld_old_set(states)
    assert np.array_equal(sample_cdf(build_cdf(p["weight"]), usel), np.arange(n_max))  # candidate n is particle n
    count = kld_count(keys)
    if name == "one_bin" or name == "distinct":
        assert count == n_max
    if name.startswith("stop_"):
        assert count == int(name[5:])
    if name in ("straddle_zero", "bin_edges"):
        assert len(np.unique(keys, axis=0)) > 100 and 2 < count
    if name == "straddle_zero":
        assert np.any((states < 0) & (keys == 0)) and np.any((states > 0) & (keys == 0))
    if name == "hash_chain":
        ts = kld_table_size(n_max)
        assert ts == 16384
        uniq = np.unique(keys, axis=0)
        assert len(uniq) >= 2000 and len(uniq) < ts // 4   # far below the table size: every probe ends
        assert np.all((kld_hash(uniq) & np.uint64(ts - 1)) == ts - 1)
        assert np.array_equal(uniq, np.unique(chain_keys(ts), axis=0))
        assert len(np.unique(uniq[:, :5], axis=0)) < len(uniq) // 20  # groups differing only in the sixth component
        assert kld_count(keys[:, :5]) < count                            # a five-component compare would stop early
    # the oracle: identity ancestors, the same count
    o = oracle.Tracker(kld=True)
    oracle.configure_like_reference(o, particle_num=n_max, max_particle_num=n_max)
    o.set_d(oracle.EPSILON, 0.2)
    o.set_vec6(oracle.BIN_SIZE, [float(BIN)] * 6)
    o.set_vec6(oracle.STEP_COV, [0.0] * 6)
    o.set_i(oracle.QUAT_SAMPLE, 0)
    o.set_particles(p)
    o.inject_draws(usel[None], np.zeros((1, n_max, 6), f32), np.ones((1, n_max), f32))
    o.resample(0)
    assert len(o.get_particles()) == count
    np.testing.assert_array_equal(o.ancestors(), np.arange(count))


# ================================================================== GPU tests
@pytest.mark.gpu
@pytest.mark.parametrize("cap,live,R", NORM_SHAPES, ids=shape_id)
def test_gpu_normalize(cap, live, R):
    """normalize_kernel reading R injected slices through raw_slot (weightPhase(2) of a sharded tracker)."""
    n = live or cap
    g, _ = make_tracker(cap, live, R=R)
    states = g.getParticles()
    for name, raw in raw_patterns(n, cap + n + R).items():
        for r, s in enumerate(raw_slices(raw, R, cap)):
            g.setRawSlice(r, s)
        for alpha in ALPHAS:
            g.setAlpha(alpha)
            g.weightPhase(2)
            want, _, wmin = ref_normalize(raw, alpha)
            got = g.getParticles()
            what = f"{name} alpha {alpha}"
            assert len(got) == n, what
            assert_flagged_equal(got["weight"], want, False, what)
            for k in STATE:
                assert np.array_equal(got[k].view(np.uint32), states[k].view(np.uint32)), (what, k)
            assert g.getFitRatio() == wmin, what


@pytest.mark.gpu
@pytest.mark.parametrize("cap,live", SHAPES, ids=shape_id)
def test_gpu_update(cap, live):
    n = live or cap
    g, _ = make_tracker(cap, live)
    for name, p in update_cases(n, cap + n).items():
        old = p[n // 2].copy()
        old["x"] += f32(0.5)
        g.setParticles(p)
        g.setResult(old, None)
        g.update()
        rep, mot, _ = ref_update(p, old)
        assert_pose_equal(g.getResult(), rep, {}, f"{name} result")
        assert_pose_equal(g.getMotion(), mot, {}, f"{name} motion")


def _compare_resample(g, o, quat, what):
    ga, oa = g.ancestors(), o.ancestors()
    assert len(ga) == len(oa), (what, len(ga), len(oa))
    np.testing.assert_array_equal(ga, oa, err_msg=what)
    gp, op = g.getParticles(), o.get_particles()
    if quat == 0:
        assert np.array_equal(gp.view(np.uint32), op.view(np.uint32)), what
    else:
        util.assert_particles_close(gp, op, 1e-6, 2e-6, None)


@pytest.mark.gpu
@pytest.mark.parametrize("kld", [False, True], ids=["fixed", "kld"])
@pytest.mark.parametrize("cap,live", SHAPES, ids=shape_id)
def test_gpu_resample(cap, live, kld):
    """cdf_kernel / alias_table_kernel / resample_kernel (and the KLD stop) against the oracle, samplers CDF, VDC and
    alias, RPY and quaternion noise, on boundary draws."""
    n = live or cap
    n_max = cap if kld else None
    g, o = make_tracker(cap, live, kld=kld, n_max=n_max)
    rng = np.random.default_rng(n + kld)
    stride = cap
    for kind in CDF_KINDS:
        w = cdf_weights(n, kind, rng)
        p = particles(n, seed=2)
        p["weight"] = w
        rep, mot = p[0].copy(), p[-1].copy()
        for k, v in zip(STATE, (0.01, -0.02, 0.005, 0.03, -0.01, 0.02)):
            mot[k] = f32(v)
        d = resample_draws(w, stride, n + len(kind))
        for sampler in (oracle.SAMPLER_CDF, oracle.SAMPLER_CDF_VDC, oracle.SAMPLER_ALIAS_PCL):
            for quat in (0, 1):
                g.setSampler(sampler); g.setQuaternionSampling(quat)
                o.set_i(oracle.SAMPLER, sampler); o.set_i(oracle.QUAT_SAMPLE, quat)
                o.set_i(oracle.PARTICLE_NUM, n)
                g.setParticles(p); o.set_particles(p)
                g.setResult(rep, mot); o.set_result(rep); o.set_motion(mot)
                g.injectDraws(*d); o.inject_draws(*d)
                g.resample(0); o.resample(0)
                _compare_resample(g, o, quat, f"{kind} sampler {sampler} quat {quat}")


@pytest.mark.gpu
@pytest.mark.parametrize("n_old,n_new", [(4000, 5000), (100000, 150)])
def test_gpu_resample_across_capacity(n_old, n_new):
    """setParticleNum across the 4096 boundary: the cluster table of a 4000-particle set, and a 150-particle draw from
    100 000."""
    for sampler in (oracle.SAMPLER_CDF, oracle.SAMPLER_CDF_VDC, oracle.SAMPLER_ALIAS_PCL):
        g, o = make_tracker(n_old, sampler=sampler, quat=0)
        w = cdf_weights(n_old, "exact", np.random.default_rng(sampler))
        p = particles(n_old, seed=3)
        p["weight"] = w
        g.setParticles(p); o.set_particles(p)
        g.setResult(p[1].copy(), p[2].copy()); o.set_result(p[1].copy())
        g.setParticleNum(n_new); o.set_i(oracle.PARTICLE_NUM, n_new)
        d = resample_draws(w, max(n_old, n_new), sampler)
        g.injectDraws(*d); o.inject_draws(*d)
        g.resample(0); o.resample(0)
        assert len(g.getParticles()) == n_new
        _compare_resample(g, o, 0, f"sampler {sampler}")


@pytest.mark.gpu
@pytest.mark.parametrize("n_max,name", KLD_CASES, ids=shape_id)
def test_gpu_kld_stop(n_max, name):
    """kld_insert_kernel / kld_stop_kernel: the particle count and every candidate against the oracle."""
    states = kld_case(n_max, name)
    p, usel = kld_old_set(states)
    g, o = make_tracker(n_max, kld=True, n_max=n_max, quat=0, epsilon=0.2, bin_size=float(BIN))
    g.setStepNoiseCovariance([0.0] * 6); o.set_vec6(oracle.STEP_COV, [0.0] * 6)
    zero = np.zeros(1, pcl.PARTICLE)[0]
    g.setParticles(p); o.set_particles(p)
    g.setResult(zero, zero); o.set_result(zero); o.set_motion(zero)
    d = (usel[None], np.zeros((1, n_max, 6), f32), motion_draws(n_max, np.random.default_rng(1))[None])
    g.injectDraws(*d); o.inject_draws(*d)
    g.resample(0); o.resample(0)
    count = kld_count(bin_keys(states))
    assert len(o.get_particles()) == count
    assert len(g.getParticles()) == count, (len(g.getParticles()), count)
    _compare_resample(g, o, 0, name)


@pytest.mark.gpu
@pytest.mark.parametrize("graph", [True, False], ids=["graph", "no_graph"])
@pytest.mark.parametrize("n", [1, 2, 1024, 4096, 4097, 8193, 100000, "kld"])
def test_gpu_compute_invariants(n, graph, monkeypatch):
    """The fused path (normalise summing the weight kernel's partials, update in the same launch) after compute():
    weights = normalise(rawWeights()), fit ratio = min(rawWeights()), result = update(getParticles()), and with one
    iteration, motion = result - previous result."""
    if not graph:
        monkeypatch.setenv("PFT_NO_GRAPH", "1")
    scene, model, centre = util.small_case(41, n_scene=3000, n_model=120)
    cloud = pcl.PointCloud(scene)
    for use_hsv in (True, False):
        for iters in (1, 2):
            kld = n == "kld"
            g, _ = util.make_pair(kld=kld, particle_num=300 if kld else n, max_particle_num=20000, use_hsv=use_hsv, iteration_num=iters)
            m = np.eye(4, dtype=f32)
            m[:3, 3] = centre
            g.setTrans(m)
            g.setReferenceCloud(model); g.setInputCloud(cloud)
            prev = None
            for frame in range(2):
                g.compute()
                what = f"hsv {use_hsv} iterations {iters} frame {frame}"
                raw, parts = g.rawWeights(), g.getParticles()
                assert len(raw) == len(parts) > 0, what
                want, flag, wmin = ref_normalize(raw, 15.0)
                assert_flagged_equal(parts["weight"], want, flag, what + " weights")
                assert g.getFitRatio() == wmin, what
                res = g.getResult()
                rep, mot, flags = ref_update(parts, prev if prev is not None else res)
                assert_pose_equal(res, rep, flags, what + " result")
                if iters == 1 and prev is not None:
                    got = g.getMotion()
                    for k in STATE:
                        assert got[k] == f32(res[k]) - f32(prev[k]), (what, k)
                prev = res.copy()
            if kld:
                assert 2 <= len(g.getParticles()) < 20000
