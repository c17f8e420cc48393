"""synth.depth_images: a rendered frame as the registered 16UC1 depth (mm) and bgr8 colour images the depth-image
ingest takes (5 bytes per pixel)."""
import numpy as np
import pytest

from pcl_tracking_b200 import synth


@pytest.mark.parametrize("sensor", [synth.KINECT2_SD, synth.KINECT2_QHD])
def test_depth_images_of_a_rendered_frame(sensor):
    w, h = sensor["width"], sensor["height"]
    pts, _ = synth.render(0, synth.default_objects(1), sensor=sensor)
    depth, bgr, K = synth.depth_images(pts, sensor)
    assert depth.shape == (h, w) and depth.dtype == np.uint16 and bgr.shape == (h, w, 3) and bgr.dtype == np.uint8
    assert depth.nbytes + bgr.nbytes == 5 * w * h
    z = pts["z"].reshape(h, w)
    finite = np.isfinite(z)
    assert np.array_equal(depth > 0, finite)  # every rendered depth lies inside 1..65535 mm
    assert np.abs(depth[finite] / 1000.0 - z[finite]).max() <= 0.0005 + 1e-6
    rgba = pts["rgba"].reshape(h, w)
    for k, shift in enumerate((0, 8, 16)):
        assert np.array_equal(bgr[..., k], ((rgba >> shift) & 0xff).astype(np.uint8))
    assert np.array_equal(K, [[sensor["f"], 0, sensor["cx"]], [0, sensor["f"], sensor["cy"]], [0, 0, 1]])
