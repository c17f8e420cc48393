"""Parity of kernel K2+K3 (scene index + weight()) with the CPU oracle, through the C ABI.

north_star bar: nearest-neighbour indices bit-exact against the exact-search coherence configuration
(ties to the lower index), particle weights within 1e-5 relative."""
import functools

import numpy as np
import pytest

import oracle
from pcl_tracking_b200 import pcl, synth
from tests import util

pytestmark = pytest.mark.gpu

W_RTOL = 1e-5


LIST_MODES = [0, 2]  # exact-NN candidate lists: never / always -- results must not depend on it


def _run_weight(seed, use_hsv, n_scene=4000, n_model=300, n_particles=48, max_dist=0.1, sigma_t=0.015, search_res=0.01, dbg=8, lists=1):
    scene, model, centre = util.small_case(seed, n_scene=n_scene, n_model=n_model)
    g, o = util.make_pair(kld=False, particle_num=n_particles, use_hsv=use_hsv, max_dist=max_dist, search_res=search_res)
    parts = util.particles_around(centre, n_particles, seed=seed + 100, sigma_t=sigma_t)
    cloud = pcl.PointCloud(scene)
    g.setReferenceCloud(model)
    g.setInputCloud(cloud)
    g.setParticles(parts)
    g.setDebugNN(dbg)
    g.setCandidateLists(lists)
    g.weight()
    assert g.indexInfo()["use_lists"] == (1 if lists == 2 else 0)
    o.set_reference(model)
    o.set_input(scene)
    o.set_particles(parts)
    o.weight(keep_nn=True)
    return g, o, scene, model


@pytest.mark.parametrize("lists", LIST_MODES)
@pytest.mark.parametrize("seed,use_hsv", [(0, False), (1, True), (2, True)])
def test_weight_matches_oracle(seed, use_hsv, lists):
    g, o, scene, model = _run_weight(seed, use_hsv, lists=lists)
    # crop box and crop count: bit-exact
    np.testing.assert_array_equal(g.aabb(), o.aabb())
    cidx, _ = o.cropped()
    assert g.croppedCount() == len(cidx)
    # nearest neighbours of the recorded particles: indices and squared distances bit-exact
    for p in range(8):
        gi, gd = g.nn(p, len(model))
        oi, od = o.nn(p, len(model))
        oi_scene = np.where(oi >= 0, cidx[np.maximum(oi, 0)], -1)
        matched = od.astype(np.float64) < 0.1 * 0.1   # the coherence only counts pairs closer than maximum_distance_
        np.testing.assert_array_equal(gi[matched], oi_scene[matched])
        np.testing.assert_array_equal(gd[matched], od[matched])
        assert np.all(gi[~matched] == -1)              # the GPU search stops at maximum_distance_
        assert matched.sum() > 0
    np.testing.assert_allclose(g.rawWeights(), o.raw_weights(), rtol=W_RTOL, atol=0)
    gp, op = g.getParticles(), o.get_particles()
    np.testing.assert_allclose(gp["weight"], op["weight"], rtol=W_RTOL, atol=1e-12)
    assert abs(float(gp["weight"].astype(np.float64).sum()) - 1.0) < 1e-4
    assert abs(g.getFitRatio() - o.fit_ratio()) <= 1e-5 * abs(o.fit_ratio())


@pytest.mark.parametrize("lists", LIST_MODES)
def test_weight_large_max_distance_all_indices_exact(lists):
    # maximum distance larger than the scene: every model point has a match; all indices must agree
    g, o, scene, model = _run_weight(5, True, n_scene=1500, n_model=120, n_particles=16, max_dist=10.0, sigma_t=0.05, dbg=16, lists=lists)
    cidx, _ = o.cropped()
    for p in range(16):
        gi, gd = g.nn(p, len(model))
        oi, od = o.nn(p, len(model))
        np.testing.assert_array_equal(gi, cidx[oi])
        np.testing.assert_array_equal(gd, od)
    np.testing.assert_allclose(g.rawWeights(), o.raw_weights(), rtol=W_RTOL)


@pytest.mark.parametrize("lists", LIST_MODES)
def test_weight_ties_go_to_lower_index(lists):
    # duplicated scene points: the same coordinates at two indices; the lower index must win
    scene, model, centre = util.small_case(7, n_scene=800, n_model=100)
    scene = np.concatenate([scene, scene[::-1]])  # every point appears twice
    g, o = util.make_pair(kld=False, particle_num=8, use_hsv=False)
    g.setCandidateLists(lists)
    parts = util.particles_around(centre, 8, seed=3)
    cloud = pcl.PointCloud(scene)
    g.setReferenceCloud(model); g.setInputCloud(cloud); g.setParticles(parts); g.setDebugNN(8); g.weight()
    o.set_reference(model); o.set_input(scene); o.set_particles(parts); o.weight(keep_nn=True)
    cidx, _ = o.cropped()
    for p in range(8):
        gi, gd = g.nn(p, len(model))
        oi, od = o.nn(p, len(model))
        m = od.astype(np.float64) < 0.01
        np.testing.assert_array_equal(gi[m], cidx[oi[m]])
        assert np.all(gi[m] < len(scene) // 2 + len(scene))  # sanity
    np.testing.assert_allclose(g.rawWeights(), o.raw_weights(), rtol=W_RTOL)


@pytest.mark.parametrize("lists", LIST_MODES)
def test_weight_coarse_and_fine_cells(lists):
    for res in (0.005, 0.02, 0.05):
        g, o, scene, model = _run_weight(11, True, n_scene=2500, n_model=150, n_particles=12, search_res=res, dbg=4, lists=lists)
        np.testing.assert_allclose(g.rawWeights(), o.raw_weights(), rtol=W_RTOL)


def test_weight_no_scene_point_in_crop():
    # scene far away from every particle: all raw weights 0 -> uniform normalised weights (A.6 fallback)
    scene, model, centre = util.small_case(3, n_scene=500, n_model=50)
    scene["x"] += 50.0
    g, o = util.make_pair(kld=False, particle_num=10, use_hsv=True)
    parts = util.particles_around(centre, 10)
    cloud = pcl.PointCloud(scene)
    g.setReferenceCloud(model); g.setInputCloud(cloud); g.setParticles(parts); g.weight()
    o.set_reference(model); o.set_input(scene); o.set_particles(parts); o.weight()
    assert g.croppedCount() == 0
    np.testing.assert_array_equal(g.rawWeights(), np.zeros(10, dtype=np.float32))
    np.testing.assert_allclose(g.getParticles()["weight"], o.get_particles()["weight"], rtol=1e-6)


def test_weight_crop_beyond_16_bit_slots():
    """A crop of more than 65 535 points: the candidate lists (16-bit slots) switch themselves off, the index is too
    large for shared memory and is read through L1/L2 -- the row-table search alone must still be exact."""
    scene, model, centre = util.small_case(21, n_scene=150000, n_model=96, spread=0.22)
    g, o = util.make_pair(kld=False, particle_num=6, use_hsv=True, oracle_nn=oracle.NN_EXACT_GRID)
    parts = util.particles_around(centre, 6, seed=5)
    cloud = pcl.PointCloud(scene)
    g.setReferenceCloud(model); g.setInputCloud(cloud); g.setParticles(parts); g.setDebugNN(6); g.setCandidateLists(2); g.weight()
    o.set_reference(model); o.set_input(scene); o.set_particles(parts); o.weight(keep_nn=True)
    cidx, _ = o.cropped()
    assert g.croppedCount() == len(cidx) and len(cidx) > 65535
    for p in range(6):
        gi, gd = g.nn(p, len(model))
        oi, od = o.nn(p, len(model))
        m = od.astype(np.float64) < 0.1 * 0.1
        np.testing.assert_array_equal(gi[m], cidx[oi[m]])
        np.testing.assert_array_equal(gd[m], od[m])
    np.testing.assert_allclose(g.rawWeights(), o.raw_weights(), rtol=W_RTOL)


def test_weight_dense_scene_long_lists():
    """3 mm point spacing against 1 cm list cells: candidate lists of 50-150 entries, some beyond the 127 of a regular
    record (extended lists) -- same nearest neighbours as brute force."""
    scene, model, centre = util.small_case(22, n_scene=60000, n_model=160, spread=0.12)
    g, o = util.make_pair(kld=False, particle_num=8, use_hsv=True, oracle_nn=oracle.NN_EXACT_GRID)
    parts = util.particles_around(centre, 8, seed=6, sigma_t=0.02)
    cloud = pcl.PointCloud(scene)
    g.setReferenceCloud(model); g.setInputCloud(cloud); g.setParticles(parts); g.setDebugNN(8); g.setCandidateLists(2); g.weight()
    assert g.indexInfo()["use_lists"] == 1
    o.set_reference(model); o.set_input(scene); o.set_particles(parts); o.weight(keep_nn=True)
    cidx, _ = o.cropped()
    for p in range(8):
        gi, gd = g.nn(p, len(model))
        oi, od = o.nn(p, len(model))
        m = od.astype(np.float64) < 0.1 * 0.1
        np.testing.assert_array_equal(gi[m], cidx[oi[m]])
        np.testing.assert_array_equal(gd[m], od[m])
    np.testing.assert_allclose(g.rawWeights(), o.raw_weights(), rtol=W_RTOL)


# ------------------------------------------------------------------ parity mode: upstream's approximate octree search
def _approx_pair(kld, n_particles, use_hsv, search_res=0.01, **kw):
    g, o = util.make_pair(kld=kld, particle_num=n_particles, use_hsv=use_hsv, oracle_nn=oracle.NN_PCL_APPROX, search_res=search_res, **kw)
    o.set_d(oracle.OCTREE_RES, search_res)
    g._si(pcl.capi.NN_MODE, pcl.capi.NN_PCL_APPROX)
    return g, o


@pytest.mark.parametrize("seed,use_hsv,search_res", [(3, True, 0.01), (4, False, 0.01), (5, True, 0.025)])
def test_weight_pcl_approx_mode_matches_oracle(seed, use_hsv, search_res):
    """PFT_NN_PCL_APPROX: the greedy octree descent of ApproxNearestPairPointCloudCoherence (ref: src/auto_tracking.cpp
    :235-236) -- same leaf, same point and same squared distance as the oracle's restatement of pcl::octree, for EVERY
    query (the approximate search has no distance cut-off), and the same weights."""
    scene, model, centre = util.small_case(seed, n_scene=5000, n_model=300)
    g, o = _approx_pair(False, 40, use_hsv, search_res)
    parts = util.particles_around(centre, 40, seed=seed + 100)
    cloud = pcl.PointCloud(scene)
    g.setReferenceCloud(model); g.setInputCloud(cloud); g.setParticles(parts); g.setDebugNN(8); g.weight()
    o.set_reference(model); o.set_input(scene); o.set_particles(parts); o.weight(keep_nn=True)
    cidx, _ = o.cropped()
    assert g.croppedCount() == len(cidx)
    for p in range(8):
        gi, gd = g.nn(p, len(model))
        oi, od = o.nn(p, len(model))
        assert np.all(oi >= 0)
        np.testing.assert_array_equal(gi, cidx[oi])
        np.testing.assert_array_equal(gd, od)
    np.testing.assert_allclose(g.rawWeights(), o.raw_weights(), rtol=W_RTOL, atol=0)
    np.testing.assert_allclose(g.getParticles()["weight"], o.get_particles()["weight"], rtol=W_RTOL, atol=1e-12)


def test_pcl_approx_mode_differs_from_exact_and_tracks():
    """The approximate search misses true neighbours (so the two modes give different weights), and a whole KLD
    compute() in the parity mode follows the oracle run in the same mode."""
    scene, model, centre = util.small_case(6, n_scene=5000, n_model=300)
    parts = util.particles_around(centre, 32, seed=9)
    cloud = pcl.PointCloud(scene)
    ge, _ = util.make_pair(kld=False, particle_num=32, use_hsv=True)
    ge.setReferenceCloud(model); ge.setInputCloud(cloud); ge.setParticles(parts); ge.setDebugNN(4); ge.weight()
    ga, _ = _approx_pair(False, 32, True)
    ga.setReferenceCloud(model); ga.setInputCloud(cloud); ga.setParticles(parts); ga.setDebugNN(4); ga.weight()
    worse = 0
    for p in range(4):
        ei, ed = ge.nn(p, len(model))
        ai, ad = ga.nn(p, len(model))
        m = ei >= 0
        assert np.all(ad[m] >= ed[m])          # never nearer than the true nearest neighbour
        worse += int((ad[m] > ed[m]).sum())
    assert worse > 0
    assert not np.array_equal(ga.rawWeights(), ge.rawWeights())

    g, o = _approx_pair(True, 100, True, max_particle_num=220)
    util.set_trans_both(g, o, centre)
    d = synth.draws(2, 220, seed=23)
    g.injectDraws(*d); o.inject_draws(*d)
    g.setReferenceCloud(model); g.setInputCloud(cloud); g.compute()
    o.set_reference(model); o.set_input(scene); o.compute()
    gp, op = g.getParticles(), o.get_particles()
    assert len(gp) == len(op)
    same = g.ancestors() == o.ancestors()
    assert same.mean() > 0.97
    for k in ("x", "y", "z", "roll", "pitch", "yaw"):
        np.testing.assert_allclose(gp[k][same], op[k][same], atol=1e-4)
    gr, orr = g.getResult(), o.get_result()
    for k in ("x", "y", "z"):
        assert abs(float(gr[k]) - float(orr[k])) < 2e-3


def test_lists_switch_off_and_on_again_on_one_tracker():
    """The candidate lists are a per-weight() decision taken on the device (enough queries for the fine cells of the crop
    box): one tracker goes through many particles (lists), a handful (row-table search inside the same kernel launch) and
    many again, against the oracle driven through the same sequence (stale slots of the crop box included)."""
    scene, model, centre = util.small_case(21, n_scene=6000, n_model=400)
    g, o = util.make_pair(kld=True, particle_num=600, max_particle_num=600, use_hsv=True, oracle_nn=oracle.NN_EXACT_GRID)
    g.setReferenceCloud(model); g.setInputCloud(pcl.PointCloud(scene))
    o.set_reference(model); o.set_input(scene)
    seen = []
    for n, seed in ((600, 3), (8, 4), (600, 5), (12, 6)):
        p = util.particles_around(centre, n, seed=seed)
        g.setParticles(p); o.set_particles(p)
        g.weight(); o.weight()
        seen.append(g.indexInfo()["use_lists"])
        np.testing.assert_array_equal(g.aabb(), o.aabb())
        np.testing.assert_allclose(g.rawWeights(), o.raw_weights(), rtol=1e-5)
        np.testing.assert_allclose(g.getParticles()["weight"], o.get_particles()["weight"], rtol=1e-5, atol=1e-12)
    assert seen == [1, 0, 1, 0]


@functools.lru_cache(maxsize=None)
def _tracked_with_timing(lists):
    """Three timed compute() calls of one fixed-N tracker (two iterations each): the kernel names of every compute(),
    the index header's list decision, and the final pose and particles as bytes."""
    scene, model, centre = util.small_case(31, n_scene=6000, n_model=400)
    t = pcl.ParticleFilterOMPTracker(16)
    pcl.configure_like_reference(t, particle_num=600, use_hsv=True, iteration_num=2)
    m = np.eye(4, dtype=np.float32)
    m[:3, 3] = centre
    t.setTrans(m); t.seed(5); t.setReferenceCloud(model); t.setCandidateLists(lists); t.enableTiming(True)
    t.setInputCloud(pcl.PointCloud(scene))
    names = []
    for _ in range(3):
        t.compute()
        names.append([n for n, _ in t.kernelTimes()])
    return names, t.indexInfo()["use_lists"], t.getResult().tobytes(), t.getParticles().tobytes()


@pytest.mark.parametrize("lists", [0, 1, 2])
def test_one_lookup_kernel_in_every_list_mode(lists):
    """Every exact-search weight() is one launch of weight_lists_kernel, with the lists off too (it then runs the row-table
    search), and the mode of the lists never changes a result: pose and particles equal bit for bit across the modes."""
    names, use_lists, pose, parts = _tracked_with_timing(lists)
    assert use_lists == (0 if lists == 0 else 1)
    for frame in names:
        assert frame.count("weight_lists_kernel") == 2  # once per iteration
        assert "weight_kernel" not in frame
    for other in (0, 1, 2):
        _, _, pose_o, parts_o = _tracked_with_timing(other)
        assert pose == pose_o and parts == parts_o
