"""The two offline drivers back to back: create_model_offline builds the object models of a recorded frame in the robot
base frame (ref: src/create_model.cpp) and writes one PCD per cluster; its files equal the Python composition of the
same steps bit for bit, and auto_tracking_offline, given them as models, tracks the objects."""
import os
import subprocess

import numpy as np
import pytest

from pcl_tracking_b200 import pcd, pcl, synth
from tests.test_gpu_model_builder import LIMITS, OBJECTS, base_from_camera, build_models, camera_from_base, np_composition, scene
from tests.test_shim import build_driver

pytestmark = pytest.mark.gpu

EXE = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "examples", "create_model_offline")


def test_create_model_offline_then_track(tmp_path):
    track_exe = build_driver()                          # make -C examples builds both drivers
    assert os.access(EXE, os.X_OK)
    pts, oid = scene(True)
    frame = tmp_path / "frame0.pcd"
    pcd.savePCDFile(frame, pts, binary=True)
    bc = base_from_camera()
    out_dir = tmp_path / "models"
    out_dir.mkdir()
    args = [EXE, str(frame)] + [repr(float(v)) for v in bc.reshape(-1)] + [repr(float(v)) for v in LIMITS] + [str(out_dir)]
    out = subprocess.run(args, capture_output=True, text=True, check=True).stdout
    lines = [tuple(int(v) for v in l.split()) for l in out.strip().splitlines()]
    # the Python composition with the reference's clustering parameters (0.02, 500, 25000)
    m_bc, m_cb = bc.astype(np.float32), camera_from_base(bc)
    _, models, clusters = build_models(pts, m_bc, m_cb, 500)
    want, ids = np_composition(pts, oid, m_bc)
    sizes = {k: int((ids == k).sum()) for k in range(OBJECTS)}
    # min 500: the objects with fewer cropped points in this frame are left out, the others are one cluster each
    assert len(clusters) == sum(s >= 500 for s in sizes.values()) and len(clusters) >= OBJECTS - 2
    assert lines == [(j, len(idx)) for j, idx in enumerate(clusters)]
    assert sorted(os.listdir(out_dir)) == sorted("%d.pcd" % j for j in range(len(clusters)))
    owners = []
    for j, (idx, model) in enumerate(zip(clusters, models)):
        got, _, _ = pcd.loadPCDFile(out_dir / ("%d.pcd" % j))
        assert np.ascontiguousarray(got).tobytes() == model.to_numpy().tobytes()
        owner = np.unique(ids[idx])
        assert len(owner) == 1
        owners.append(int(owner[0]))
    # those PCDs are auto_tracking_offline's models: it follows every object over two frames
    frames = []
    for f in range(2):
        p = tmp_path / ("frame%d.raw" % f)
        p.write_bytes(synth.to_pcl32(synth.render(f, synth.default_objects(OBJECTS, seed=3))[0]).tobytes())
        frames.append(str(p))
    model_arg = ",".join(str(out_dir / ("%d.pcd" % j)) for j in range(len(clusters)))
    track = subprocess.run([track_exe, model_arg, "11"] + frames, capture_output=True, text=True, check=True).stdout
    rows = [l.split() for l in track.strip().splitlines()]
    assert len(rows) == 2 * len(clusters)
    last_pts, last_oid = synth.render(1, synth.default_objects(OBJECTS, seed=3))
    for j, owner in enumerate(owners):
        pose = np.array([float(v) for v in rows[len(clusters) + j][2:5]])
        sel = (last_oid == owner) & np.isfinite(last_pts["x"])
        centre = np.array([last_pts[k][sel].astype(np.float64).mean() for k in ("x", "y", "z")])
        assert np.linalg.norm(pose - centre) < 0.03, (j, owner, pose, centre)
