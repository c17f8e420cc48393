"""bench.py --dump-outputs writes what the last timed step of the headline workload computed, and --steps is the number
of timed steps: two runs that track the same seven frames (3 warm-up + 4 timed, 5 warm-up + 2 timed) dump the same
outputs, and the dumped cloud is the downsampled frame shown at step 6."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out, steps, warmup):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", str(warmup),
                        "--also", "none", "--no-cpu-baseline", "--dump-outputs", str(out)],
                       capture_output=True, text=True, cwd=ROOT, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [json.loads(ln) for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1 and lines[0]["steps"] == steps and lines[0]["warmup"] == warmup
    return {n: np.load(os.path.join(out, n + ".npy")) for n in ("downsampled_cloud", "result", "particles")}


@pytest.mark.gpu
def test_bench_dumps_the_outputs_of_its_last_timed_step(tmp_path):
    import oracle
    from pcl_tracking_b200 import synth
    a = _bench(tmp_path / "a", steps=4, warmup=3)
    b = _bench(tmp_path / "b", steps=2, warmup=5)
    assert a["downsampled_cloud"].dtype == np.float32 and a["downsampled_cloud"].shape[1] == 7
    assert a["result"].shape == (1, 8) and a["particles"].shape == (1000, 8)
    assert abs(float(a["particles"][:, 7].astype(np.float64).sum()) - 1.0) < 1e-4
    for k in a:
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    frame = synth.render(4, synth.default_objects(1))[0]  # ping-pong order over 6 frames: step 6 shows frame 4
    ref = oracle.voxel_grid_exact(frame, 0.01, 2, 0.0, 10.0)
    rgba = np.ascontiguousarray(ref["rgba"]).view(np.uint8).reshape(-1, 4)[:, [2, 1, 0, 3]]
    want = np.column_stack([ref["x"], ref["y"], ref["z"], rgba.astype(np.float32)])
    np.testing.assert_array_equal(a["downsampled_cloud"], want)
