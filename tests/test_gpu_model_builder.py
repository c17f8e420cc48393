"""The model builder (ref: src/create_model.cpp) end to end on the device, in the robot base frame: removeZeroPoints,
transformPointCloud into the base frame, the segm_limits crop (three PassThroughs) or the plane variant's RANSAC
(ref: src/create_model_planar_segmentation.cpp:157-174), Euclidean clustering, and every cluster moved back to the
camera frame -- the models the trackers then follow.  The base frame is the synthetic table's: origin at its point,
axes u, v, n (synth.table_frame()), so the table lies at z = 0 and the objects stand on it."""
import numpy as np
import pytest

from pcl_tracking_b200 import pcl, synth
from tests.test_gpu_compute import _tracker_for
from tests.test_gpu_transform import np_keep_nonzero, np_transform, same_bits

pytestmark = pytest.mark.gpu

# segm_limits in the base frame (x = u, y = v, z = n): the part of the table the objects stand on, from 1.5 cm above it
LIMITS = (-0.6, 0.6, -0.4, 0.4, 0.015, 0.4)
OBJECTS = 8


def scene(noise):
    return synth.render(0, synth.default_objects(OBJECTS, seed=3), noise=noise)


def base_from_camera():
    """The double 3x4 [R|t] tf would give: p_base = R (p_cam - P) with the rows of R the table axes u, v, n."""
    u, v, n = synth.table_frame()
    R = np.stack([u, v, n])
    m = np.zeros((3, 4))
    m[:, :3], m[:, 3] = R, -(R @ synth._TABLE_P)
    return m


def camera_from_base(bc):
    """Its inverse (R^T, -R^T t) computed in double, each row of R^T t summed left to right, then rounded to float --
    as examples/create_model_offline.cpp computes it."""
    m = np.zeros((3, 4), dtype=np.float32)
    for r in range(3):
        for c in range(3):
            m[r, c] = np.float32(bc[c, r])
        m[r, 3] = np.float32(-((float(bc[0, r]) * float(bc[0, 3]) + float(bc[1, r]) * float(bc[1, 3])) + float(bc[2, r]) * float(bc[2, 3])))
    return m


def np_crop(pts, fields, limits):
    """Sequential PassThroughs: finite points with lo <= value <= hi (float32 limits), order preserving."""
    keep = np.ones(len(pts), dtype=bool)
    for k, f in enumerate(fields):
        lo, hi = np.float32(limits[2 * k]), np.float32(limits[2 * k + 1])
        x, y, z = pts["x"], pts["y"], pts["z"]
        fin = np.isfinite(x) & np.isfinite(y) & np.isfinite(z)
        with np.errstate(invalid="ignore"):
            keep &= fin & (pts[f] >= lo) & (pts[f] <= hi)
    return keep


def device_crop(cloud, fields, limits):
    for k, f in enumerate(fields):
        pt = pcl.PassThrough()
        pt.setFilterFieldName(f)
        pt.setFilterLimits(limits[2 * k], limits[2 * k + 1])
        pt.setInputCloud(cloud)
        cloud = pt.filter()
    return cloud


def clusters_of(cloud, min_size):
    ec = pcl.EuclideanClusterExtraction()
    ec.setClusterTolerance(0.02); ec.setMinClusterSize(min_size); ec.setMaxClusterSize(25000)
    ec.setInputCloud(cloud)
    return ec, ec.extract()


def build_models(pts, m_bc, m_cb, min_size):
    """The passthrough variant on the device.  Returns (cropped base-frame cloud, its numpy composition, the object id of
    each of its points, clusters, camera-frame model clouds)."""
    nz = pcl.removeZeroPoints(pcl.PointCloud(pts))
    base = pcl.transformPointCloud(nz, m_bc)
    crop = device_crop(base, "xyz", LIMITS)
    ec, clusters = clusters_of(crop, min_size)
    models = [pcl.transformPointCloud(ec.cluster_cloud(k), m_cb) for k in range(len(clusters))]
    return crop, models, clusters


def np_composition(pts, oid, m_bc):
    keep = np_keep_nonzero(pts)
    p = np_transform(pts[keep], m_bc)
    crop = np_crop(p, "xyz", LIMITS)
    return p[crop], oid[keep][crop]


@pytest.mark.parametrize("noise", [False, True])
def test_passthrough_variant(noise):
    pts, oid = scene(noise)
    bc = base_from_camera()
    m_bc, m_cb = bc.astype(np.float32), camera_from_base(bc)
    crop, models, clusters = build_models(pts, m_bc, m_cb, 200)
    want, ids = np_composition(pts, oid, m_bc)
    assert same_bits(crop.to_numpy(), want)
    # the limits hold no table or wall point, and some of every object
    assert (ids < 0).sum() == 0 and set(np.unique(ids)) == set(range(OBJECTS))
    assert len(clusters) == OBJECTS
    if not noise:
        # every object is exactly one cluster and every cluster one whole object: the clusters are the objects' cropped
        # points, ranked by size (ties: lower first index)
        groups = sorted((np.flatnonzero(ids == k) for k in range(OBJECTS)), key=lambda g: (-len(g), g[0]))
        for idx, g in zip(clusters, groups):
            assert np.array_equal(idx, g)
    else:
        owners = [np.unique(ids[idx]) for idx in clusters]
        assert all(len(o) == 1 for o in owners)
        assert sorted(int(o[0]) for o in owners) == list(range(OBJECTS))
    # the model clouds: the numpy composition of the same steps, bit for bit
    for idx, model in zip(clusters, models):
        assert same_bits(model.to_numpy(), np_transform(want[idx], m_cb))
    # trackers built from them stay on their objects (as the C5 test of the ground-truth models)
    vg = pcl.ApproximateVoxelGrid()
    vg.setLeafSize(0.01); vg.setPassThrough("z", 0.0, 10.0); vg.setInputCloud(pcl.PointCloud(pts))
    ds = vg.filter()
    trackers = []
    for k, model in enumerate(models):
        prepared, c = pcl.prepare_model(model, 0.01)
        t = _tracker_for(prepared, c, kld=False, n=200, nmax=200, use_hsv=True, seed=7 + k)
        t.setInputCloud(ds)
        trackers.append(t)
    for _ in range(2):
        pcl.compute_batch(trackers)
    for t, model in zip(trackers, models):
        m = model.to_numpy()
        centre = np.array([m["x"].mean(), m["y"].mean(), m["z"].mean()])
        assert np.linalg.norm(t.getResultBox()["centroid"] - centre) < 0.03


def subsequence_index(whole, part):
    """Positions of the points of `part` in `whole`, of which it is an order-preserving subsequence."""
    w, p = np.ascontiguousarray(whole).view("V16"), np.ascontiguousarray(part).view("V16")
    idx, j = [], 0
    for i in range(len(w)):
        if j < len(p) and w[i] == p[j]:
            idx.append(i)
            j += 1
    assert j == len(p)
    return np.asarray(idx, dtype=np.int64)


@pytest.mark.parametrize("noise", [False, True])
def test_planar_variant(noise):
    """The plane variant: the z PassThrough replaced by SACSegmentation(plane, RANSAC, 1000 iterations, 0.015) and the
    negative ExtractIndices.  Every object ends in exactly one cluster, each cluster is part of one object, and nothing
    of the table is left in any cluster."""
    pts, oid = scene(noise)
    m_bc = base_from_camera().astype(np.float32)
    nz = pcl.removeZeroPoints(pcl.PointCloud(pts))
    crop = device_crop(pcl.transformPointCloud(nz, m_bc), "xy", LIMITS)
    keep = np_keep_nonzero(pts)
    p = np_transform(pts[keep], m_bc)
    in_xy = np_crop(p, "xy", LIMITS)
    assert same_bits(crop.to_numpy(), p[in_xy])
    ids = oid[keep][in_xy]
    seg = pcl.SACSegmentation()
    seg.setModelType("SACMODEL_PLANE"); seg.setMethodType("SAC_RANSAC")
    seg.setMaxIterations(1000); seg.setDistanceThreshold(0.015)
    seg.setInputCloud(crop)
    coeff, n_in = seg.segment()
    assert abs(abs(coeff[2]) - 1.0) < 1e-3                          # the table: z = 0 in the base frame
    rest = seg.rest.to_numpy()
    rest_ids = ids[subsequence_index(crop.to_numpy(), rest)]
    _, clusters = clusters_of(seg.rest, 200)
    owners = [np.unique(rest_ids[idx]) for idx in clusters]
    assert all(len(o) == 1 and o[0] >= 0 for o in owners)           # one object each, no table or wall point
    assert sorted(int(o[0]) for o in owners) == list(range(OBJECTS))  # every object exactly once
