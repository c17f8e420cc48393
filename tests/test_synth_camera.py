"""synth.render(camera=...): the same table, wall and objects ray-cast from another calibrated viewpoint, the input of
the multi-camera ingest tests."""
import hashlib

import numpy as np

from pcl_tracking_b200 import synth


def _world(pts, camera):
    xyz = np.stack([pts["x"], pts["y"], pts["z"]], axis=1).astype(np.float64)
    return xyz @ np.asarray(camera[0]).T + np.asarray(camera[1])


def test_side_view_table_points_lie_on_the_table_plane():
    cam = synth.side_camera()
    R = cam[0]
    assert np.allclose(R.T @ R, np.eye(3), atol=1e-12) and abs(np.linalg.det(R) - 1.0) < 1e-12
    pts, oid = synth.render(0, synth.default_objects(1), camera=cam, noise=False, holes=0)
    finite = np.isfinite(pts["z"])
    assert finite.any() and (pts["z"][finite] > 0).all()
    w = _world(pts, cam)
    u, v, n = synth.table_frame()
    rel = w - synth._TABLE_P
    # background hits are the table rectangle or the wall (world z = 3.5); near ones only, where fp32 keeps 1e-6 m
    table = finite & (oid == -1) & (pts["z"] < 3.0) & (np.abs(w[:, 2] - 3.5) > 1e-5)
    assert table.sum() > 10000
    assert np.abs(rel[table] @ n).max() <= 1e-6
    assert (np.abs(rel[table] @ u) < 0.85 + 1e-6).all() and (np.abs(rel[table] @ v) < 0.60 + 1e-6).all()
    # the object is seen from the side too, and sits above the table
    obj = finite & (oid == 0)
    assert obj.sum() > 1000
    assert (rel[obj] @ n > -1e-6).all()


def test_side_view_matches_a_transformed_render_of_the_same_scene():
    # a point of the object seen by both cameras: the object's world centre is the same whichever camera looks at it
    objs = synth.default_objects(1)
    cam = synth.side_camera()
    R, c = synth.object_pose(objs[0], 3)
    pts, oid = synth.render(3, objs, camera=cam, noise=False, holes=0)
    w = _world(pts, cam)[oid == 0]
    half = objs[0]["size"] / 2
    local = (w - c) @ R  # box frame
    assert (np.abs(local) <= half + 1e-6).all()
    assert (np.abs(np.abs(local) - half) <= 1e-6).any(axis=1).all()  # on the box's surface


def test_default_camera_output_unchanged():
    # sha256 of (points, object ids) of the default viewpoint as rendered before render() took a camera: bench.py and
    # the existing tests depend on these frames
    cases = [(0, 1, synth.KINECT2_SD, "f4e28f1f50ca35a80566d618319c3339524c3110f253ab32811edad587bc32bc"),
             (2, 3, synth.KINECT2_QHD, "a425a93b83551d0ebdeb693c757a848d2730bcee6b7dca8a9c917bdd2c38a23f")]
    for frame, k, sensor, want in cases:
        for kw in ({}, {"camera": None}):
            pts, oid = synth.render(frame, synth.default_objects(k), sensor=sensor, **kw)
            assert hashlib.sha256(pts.tobytes() + oid.tobytes()).hexdigest() == want, (frame, k, kw)
