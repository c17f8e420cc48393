"""One object per GPU: trackers on contexts other than the sensor's take the scene that context 0 downsampled
(pft_tracker_set_input_cloud with a cloud of another context).  Each destination context reads one replica of the
scene, refreshed by one fan-out launch per frame.  Results must equal the same trackers on context 0 bit for bit.
The extra contexts sit on real second devices when there are any, else on device 0 (a context of its own each)."""
import gc
import os
import subprocess

import numpy as np
import pytest

from pcl_tracking_b200 import pcl, synth

pytestmark = pytest.mark.gpu

N_OBJ, FRAMES = 3, 6


def _device(k):
    import torch
    n = torch.cuda.device_count()
    return k % n if n >= 2 else 0


def _frames(n=FRAMES):
    objs = synth.default_objects(N_OBJ, seed=3)
    out = [synth.render(f, objs) for f in range(n)]
    return [p for p, _ in out], out[0][1]


class Scene:
    """The sensor's side on context `ctx`: raw frames in HBM, downsampled into ONE cloud refilled in place."""

    def __init__(self, ctx, frames, zmax=None):
        self.ctx = ctx
        self.raw = [pcl.PointCloud(f, ctx=ctx) for f in frames]
        self.ds = pcl.PointCloud(ctx=ctx)
        self.vg = pcl.ApproximateVoxelGrid(ctx=ctx)
        self.vg.setLeafSize(0.01, 0.01, 0.01)
        self.zmax = zmax

    def frame(self, f):
        self.vg.setPassThrough("z", 0.0, self.zmax[f] if self.zmax else 10.0)
        self.vg.setInputCloud(self.raw[f])
        self.vg.filter(self.ds)
        return self.ds


def _trackers(ctxs, kld, frames, oid0, sensor_ctx):
    """Tracker k (object k % N_OBJ) on ctxs[k]; the models are prepared on the sensor's context."""
    ts = []
    for k, ctx in enumerate(ctxs):
        model, c = pcl.prepare_model(pcl.PointCloud(synth.model_points(frames[0], oid0, k % N_OBJ), ctx=sensor_ctx), 0.01)
        t = (pcl.KLDAdaptiveParticleFilterOMPTracker if kld else pcl.ParticleFilterOMPTracker)(16, ctx=ctx)
        if kld:
            pcl.configure_like_reference(t, particle_num=150, max_particle_num=220, use_hsv=True, iteration_num=2)
        else:
            pcl.configure_like_reference(t, particle_num=180, use_hsv=True, iteration_num=2)
        m = np.eye(4, dtype=np.float32)
        m[:3, 3] = c
        t.setTrans(m)
        t.seed(1234 + k)
        t.setReferenceCloud(model)
        t.setMinIndices(model.size() // 2)
        ts.append(t)
    return ts


def _state(ts):
    return [(t.getParticles().copy(), t.rawWeights().copy(), np.array(t.getResult().tolist(), dtype=np.float32)) for t in ts]


def _step(ts, cloud, batch):
    for t in ts:
        t.setInputCloud(cloud)
    if batch:
        pcl.compute_batch(ts)
    else:
        for t in ts:
            t.compute()


def _run(ctxs, kld, batch, sensor_ctx, provider, n=FRAMES):
    frames, oid0 = _frames()
    ts = _trackers(ctxs, kld, frames, oid0, sensor_ctx)
    out = []
    for f in range(n):
        _step(ts, provider(f), batch)
        out.append(_state(ts))
    return ts, out


def _assert_same(got, want):
    for f, (g, w) in enumerate(zip(got, want)):
        for k, (gk, wk) in enumerate(zip(g, w)):
            for j, name in enumerate(("particles", "raw weights", "result")):
                assert np.array_equal(gk[j].view(np.uint32), wk[j].view(np.uint32)), "%s of tracker %d differ: frame %d" % (name, k, f)


@pytest.mark.parametrize("kld", [False, True])
def test_round_robin_placement_equals_one_context(kld):
    frames, _ = _frames()
    ctx0 = pcl.Context(0)
    scene = Scene(ctx0, frames)
    _, want = _run([ctx0] * N_OBJ, kld, False, ctx0, scene.frame)
    ctxs = [ctx0, pcl.Context(_device(1)), pcl.Context(_device(2))]
    for batch in (False, True):
        ts, got = _run(ctxs, kld, batch, ctx0, scene.frame)
        _assert_same(got, want)
        assert all(t.graphReplays() > 0 for t in ts)


def test_one_fanout_per_destination_context_and_frame():
    frames, _ = _frames()
    ctx0 = pcl.Context(0)
    scene = Scene(ctx0, frames)
    ctx_b = pcl.Context(_device(1))

    def per_frame(ctxs, batch):
        fr, oid0 = _frames()
        ts = _trackers(ctxs, False, fr, oid0, ctx0)
        for f in range(3):  # graphs captured
            _step(ts, scene.frame(f), batch)
        ctx0.synchronize()
        deltas = []
        for f in range(3, 6):
            c0 = pcl.kernel_launch_count()
            _step(ts, scene.frame(f), batch)
            deltas.append(pcl.kernel_launch_count() - c0)
        c0 = pcl.kernel_launch_count()
        _step(ts, scene.ds, batch)  # the scene did not change: nothing to copy
        same = pcl.kernel_launch_count() - c0
        c0 = pcl.kernel_launch_count()
        scene.frame(5)
        refill = pcl.kernel_launch_count() - c0
        return deltas, same, refill

    for batch in (False, True):
        ref, ref_same, refill = per_frame([ctx0] * 4, batch)
        placed, placed_same, _ = per_frame([ctx0, ctx_b, ctx_b, ctx_b], batch)
        assert [p - r for p, r in zip(placed, ref)] == [1, 1, 1], (placed, ref)
        assert placed_same == ref_same == ref[0] - refill, (placed_same, ref_same, ref, refill)


def test_replicas_follow_their_source():
    """A shrinking scene refilled in place, a scene filled by an asynchronous upload, and a destroyed source replaced by a
    new cloud (whose storage may sit where the old one was) all reach the other contexts."""
    frames, _ = _frames()
    ctx0 = pcl.Context(0)
    zmax = [10.0, 3.0, 2.2, 1.8, 1.6, 10.0]
    shrink = Scene(ctx0, frames, zmax)
    ds_host = [shrink.frame(f).to_numpy() for f in range(FRAMES)]
    pinned = [pcl.PinnedBuffer.of(d) for d in ds_host]
    async_cloud = pcl.PointCloud(ctx=ctx0)

    def by_async_upload(f):
        async_cloud.upload_raw_async(pinned[f].ptr, len(ds_host[f]))
        return async_cloud

    fresh = {}

    def new_cloud_each_frame(f):
        fresh.pop("c", None)
        gc.collect()
        fresh["c"] = pcl.PointCloud(ds_host[f], ctx=ctx0)
        return fresh["c"]

    placed = [pcl.Context(_device(1)), pcl.Context(_device(2)), pcl.Context(_device(1))]
    for provider in (shrink.frame, by_async_upload, new_cloud_each_frame):
        _, want = _run([ctx0] * N_OBJ, True, False, ctx0, provider)
        ts, got = _run(placed, True, False, ctx0, provider)
        _assert_same(got, want)
        _step(ts, None, False)


@pytest.mark.parametrize("source_first", [True, False])
def test_destroy_order(source_first):
    frames, oid0 = _frames(2)
    ctx0, ctx_b = pcl.Context(0), pcl.Context(_device(1))
    scene = Scene(ctx0, frames)
    ts = _trackers([ctx_b, ctx_b], False, frames, oid0, ctx0)
    _step(ts, scene.frame(0), False)
    _step(ts, scene.frame(1), True)
    _step(ts, None, False)  # (no tracker may outlive its context below)
    if source_first:
        del scene
        gc.collect()
        del ts
        gc.collect()
        ctx_b.close()
    else:
        del ts
        gc.collect()
        ctx_b.close()
        del scene
        gc.collect()
    ctx0.synchronize()


def test_sharded_tracker_refuses_a_cloud_of_another_context():
    frames, oid0 = _frames(1)
    ctx0, ctx_b = pcl.Context(0), pcl.Context(_device(1))
    t = pcl.ParticleFilterOMPTracker(16, ctx=ctx_b)
    t.setShard(2, 0)
    with pytest.raises(pcl.PftError) as e:
        t.setInputCloud(pcl.PointCloud(frames[0], ctx=ctx0))
    assert e.value.code == pcl.capi.ERR_INVALID


def test_set_devices_tracker_with_a_foreign_input():
    import torch
    devices = [0, 1] if torch.cuda.device_count() >= 2 else [0, 0]
    frames, _ = _frames()
    ctx0 = pcl.Context(0)
    scene = Scene(ctx0, frames)
    _, want = _run([ctx0], True, False, ctx0, scene.frame)
    fr, oid0 = _frames()
    model, c = pcl.prepare_model(pcl.PointCloud(synth.model_points(fr[0], oid0, 0), ctx=ctx0), 0.01)
    t = pcl.KLDAdaptiveParticleFilterOMPTracker(16, ctx=pcl.Context(devices[0]))
    t.setDevices(devices)
    pcl.configure_like_reference(t, particle_num=150, max_particle_num=220, use_hsv=True, iteration_num=2)
    m = np.eye(4, dtype=np.float32)
    m[:3, 3] = c
    t.setTrans(m)
    t.seed(1234)
    t.setReferenceCloud(model)
    t.setMinIndices(model.size() // 2)
    got = []
    for f in range(FRAMES):
        _step([t], scene.frame(f), False)
        got.append(_state([t]))
    _assert_same(got, want)
    assert t.graphReplays() > 0


def test_offline_driver_places_objects_on_devices(tmp_path):
    from tests.test_shim import build_driver
    import torch
    exe = build_driver()
    frames, oid0 = _frames(3)
    models = []
    for k in range(2):
        p = tmp_path / ("model%d.raw" % k)
        p.write_bytes(synth.to_pcl32(synth.model_points(frames[0], oid0, k)).tobytes())
        models.append(str(p))
    names = []
    for k, f in enumerate(frames):
        p = tmp_path / ("frame%d.raw" % k)
        p.write_bytes(synth.to_pcl32(f).tobytes())
        names.append(str(p))
    cmd = [exe, ",".join(models), "4242"] + names
    env = {k: v for k, v in os.environ.items() if k not in ("PFT_DEVICES", "PFT_OBJECT_DEVICES")}
    one = subprocess.run(cmd, capture_output=True, text=True, check=True, env=env).stdout
    assert len(one.strip().splitlines()) == 2 * len(frames)
    devs = "0,1" if torch.cuda.device_count() >= 2 else "0,0"
    placed = subprocess.run(cmd, capture_output=True, text=True, check=True, env=dict(env, PFT_OBJECT_DEVICES=devs)).stdout
    assert placed == one
    both = subprocess.run(cmd, capture_output=True, text=True, env=dict(env, PFT_OBJECT_DEVICES=devs, PFT_DEVICES=devs))
    assert both.returncode != 0
