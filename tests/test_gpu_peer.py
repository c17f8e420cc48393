"""NVLink peer exchange (pft_tracker_peer_*): R processes, one tracker rank each, exchange the crop box and
the raw weights of weight() through CUDA-IPC windows written by the producing kernels themselves.  The
sharded run must equal the unsharded one bit for bit, over several compute() calls (CUDA-graph replays
included).  With fewer GPUs than ranks the ranks share GPU 0 (the driver time-slices the processes), so the
test also runs on a one-GPU box."""
import multiprocessing as mp
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N_PART, N_MAX, FRAMES = 101, 160, 4


def _coherence(parity):
    """The default exact search, or the parity search (upstream's greedy octree descent)."""
    from pcl_tracking_b200 import pcl
    if not parity:
        return pcl.NearestPairPointCloudCoherence()
    c = pcl.ApproxNearestPairPointCloudCoherence()
    c.setPclApproximateSearch(True)
    return c


def _tracker(kld, shard=None, device=0, parity=False):
    from pcl_tracking_b200 import pcl
    from tests import util
    ctx = pcl.Context(device)
    scene, model, centre = util.small_case(77, n_scene=4000, n_model=260)
    g = (pcl.KLDAdaptiveParticleFilterOMPTracker if kld else pcl.ParticleFilterOMPTracker)(16, ctx=ctx)
    pcl.configure_like_reference(g, coherence_cls=lambda: _coherence(parity), particle_num=N_PART, max_particle_num=N_MAX,
                                 use_hsv=True, iteration_num=2)
    if kld:
        g.setEpsilon(0.2)
        g.setBinSize([0.1] * 6)
    m = np.eye(4, dtype=np.float32)
    m[:3, 3] = centre
    g.setTrans(m)
    g.seed(99)
    if shard:
        g.setShard(*shard)
    g.setReferenceCloud(model)
    cloud = pcl.PointCloud(scene, ctx=ctx)
    g.setInputCloud(cloud)
    return ctx, g, cloud


def _run(g):
    out = []
    for _ in range(FRAMES):
        g.compute()
        out.append((g.getParticles().copy(), g.rawWeights().copy(), np.array(g.getResult().tolist(), dtype=np.float32)))
    return out


def _rank_main(rank, nranks, kld, conns, result_q):
    try:
        sys.path.insert(0, ROOT)
        import torch  # noqa: F401  (device count)
        device = rank if torch.cuda.device_count() >= nranks else 0
        ctx, g, cloud = _tracker(kld, (nranks, rank), device)
        mine = g.peerExport()
        # all-gather of the handles through the parent
        conns[rank].send(mine)
        handles = conns[rank].recv()
        g.peerAttach(handles)
        conns[rank].send("attached")
        assert conns[rank].recv() == "go"
        out = _run(g)
        replays = g.graphReplays()
        g.peerDetach()
        result_q.put((rank, out, replays, None))
    except Exception as e:  # pragma: no cover
        import traceback
        result_q.put((rank, None, 0, traceback.format_exc() + repr(e)))


@pytest.mark.parametrize("nranks,kld", [(2, False), (3, True)])
def test_peer_exchange_equals_unsharded(nranks, kld):
    mpc = mp.get_context("spawn")
    pipes = [mpc.Pipe() for _ in range(nranks)]
    q = mpc.Queue()
    procs = [mpc.Process(target=_rank_main, args=(r, nranks, kld, [p[1] for p in pipes], q)) for r in range(nranks)]
    for p in procs:
        p.start()
    try:
        handles = []
        for r in range(nranks):
            assert pipes[r][0].poll(180), "rank %d did not export its window" % r
            handles.append(pipes[r][0].recv())
        for r in range(nranks):
            pipes[r][0].send(handles)
        for r in range(nranks):
            assert pipes[r][0].poll(120) and pipes[r][0].recv() == "attached"
        for r in range(nranks):
            pipes[r][0].send("go")
        results = {}
        for _ in range(nranks):
            rank, out, replays, err = q.get(timeout=300)
            assert err is None, "rank %d failed:\n%s" % (rank, err)
            results[rank] = (out, replays)
    finally:
        for p in procs:
            p.join(timeout=30)
            if p.is_alive():
                p.kill()
    # the unsharded run, in this process
    ctx, g, cloud = _tracker(kld)
    want = _run(g)
    for rank in range(nranks):
        out, replays = results[rank]
        assert replays >= 1, "steady-state frames must replay the CUDA graph with the peer exchange captured in it"
        for f in range(FRAMES):
            assert np.array_equal(out[f][0].view(np.uint32), want[f][0].view(np.uint32)), "particles differ: rank %d frame %d" % (rank, f)
            assert np.array_equal(out[f][1].view(np.uint32), want[f][1].view(np.uint32)), "raw weights differ: rank %d frame %d" % (rank, f)
            assert np.array_equal(out[f][2].view(np.uint32), want[f][2].view(np.uint32)), "result differs: rank %d frame %d" % (rank, f)


# ---------------------------------------------------------------- scene distribution by peer stores (pft_cloud_peer_*)
SCENE_FRAMES = 3


def _scene_frame(k):
    from pcl_tracking_b200 import pcl
    rng = np.random.default_rng(500 + k)
    n = 3000 + 700 * k  # the point count changes from frame to frame (it travels in the header)
    pts = np.zeros(n, dtype=pcl.POINT)
    xyz = rng.uniform(-0.5, 0.5, size=(n, 3)).astype(np.float32) + np.array([0, 0, 1.5], dtype=np.float32)
    pts["x"], pts["y"], pts["z"] = xyz[:, 0], xyz[:, 1], xyz[:, 2]
    c = rng.integers(0, 256, (n, 3)).astype(np.uint32)
    pts["rgba"] = (255 << 24) | (c[:, 0] << 16) | (c[:, 1] << 8) | c[:, 2]
    return pts


def _scene_rank_main(rank, nranks, track, conns, result_q):
    try:
        sys.path.insert(0, ROOT)
        import torch  # noqa: F401
        from pcl_tracking_b200 import pcl
        device = rank if torch.cuda.device_count() >= nranks else 0
        if track:
            ctx, g, cloud0 = _tracker(False, (nranks, rank), device)
            conns[rank].send(g.peerExport())
            g.peerAttach(conns[rank].recv())
            scene0 = cloud0.to_numpy()
        else:
            ctx = pcl.Context(device)
        ds = pcl.PointCloud(ctx=ctx)
        conns[rank].send(ds.peerExport(8192))
        ds.peerAttach(conns[rank].recv(), rank)
        conns[rank].send("attached")
        assert conns[rank].recv() == "go"
        out = []
        vg = pcl.ApproximateVoxelGrid(ctx=ctx)
        vg.setLeafSize(0.02, 0.02, 0.02)
        vg.setPassThrough("z", 0.0, 10.0)
        for k in range(FRAMES if track else SCENE_FRAMES):
            if rank == 0:  # the rank that owns the sensor
                if track:
                    ds.upload(scene0)
                else:
                    vg.setInputCloud(pcl.PointCloud(_scene_frame(k), ctx=ctx))
                    vg.filter(ds)
            ds.peerBroadcast(0)
            if track:
                g.setInputCloud(ds)
                g.compute()
                out.append((g.getParticles().copy(), g.rawWeights().copy(), np.array(g.getResult().tolist(), dtype=np.float32)))
            else:
                out.append(ds.to_numpy().copy())
                conns[rank].send("read %d" % k)  # (no tracker loop here: the parent keeps the root from refilling the cloud early)
                assert conns[rank].recv() == "next"
        if track:
            g.peerDetach()
        ds.peerDetach()
        result_q.put((rank, out, None))
    except Exception as e:  # pragma: no cover
        import traceback
        result_q.put((rank, None, traceback.format_exc() + repr(e)))


def _exchange(pipes, nranks, what):
    got = []
    for r in range(nranks):
        assert pipes[r][0].poll(180), "rank %d did not send its %s" % (r, what)
        got.append(pipes[r][0].recv())
    return got


@pytest.mark.parametrize("nranks,track", [(2, False), (3, False), (2, True)])
def test_scene_peer_broadcast(nranks, track):
    """One rank fills the downsampled scene, its push kernel stores it into every rank's cloud: every rank reads the
    root's bytes (point count included), and a sharded tracker fed this way equals the unsharded run bit for bit."""
    mpc = mp.get_context("spawn")
    pipes = [mpc.Pipe() for _ in range(nranks)]
    q = mpc.Queue()
    procs = [mpc.Process(target=_scene_rank_main, args=(r, nranks, track, [p[1] for p in pipes], q)) for r in range(nranks)]
    for p in procs:
        p.start()
    try:
        for what in (["tracker window"] if track else []) + ["cloud handles"]:
            handles = _exchange(pipes, nranks, what)
            for r in range(nranks):
                pipes[r][0].send(handles)
        assert _exchange(pipes, nranks, "attach") == ["attached"] * nranks
        for r in range(nranks):
            pipes[r][0].send("go")
        if not track:
            for k in range(SCENE_FRAMES):
                assert _exchange(pipes, nranks, "frame") == ["read %d" % k] * nranks
                for r in range(nranks):
                    pipes[r][0].send("next")
        results = {}
        for _ in range(nranks):
            rank, out, err = q.get(timeout=300)
            assert err is None, "rank %d failed:\n%s" % (rank, err)
            results[rank] = out
    finally:
        for p in procs:
            p.join(timeout=30)
            if p.is_alive():
                p.kill()
    if track:
        ctx, g, cloud = _tracker(False)
        want = _run(g)
        for rank in range(nranks):
            for f in range(FRAMES):
                for j, name in enumerate(("particles", "raw weights", "result")):
                    assert np.array_equal(results[rank][f][j].view(np.uint32), want[f][j].view(np.uint32)), "%s differ: rank %d frame %d" % (name, rank, f)
    else:
        for k in range(SCENE_FRAMES):
            assert len(results[0][k]) > 100
            for rank in range(1, nranks):
                assert results[rank][k].tobytes() == results[0][k].tobytes(), "scene %d differs on rank %d" % (k, rank)
        assert len({len(results[0][k]) for k in range(SCENE_FRAMES)}) > 1


def test_exported_cloud_refuses_to_grow():
    from pcl_tracking_b200 import pcl
    ctx = pcl.Context(0)
    c = pcl.PointCloud(ctx=ctx)
    c.peerExport(1000)
    c.upload(_scene_frame(0)[:900])
    with pytest.raises(pcl.PftError):
        c.upload(_scene_frame(0)[:2000])
    c.peerDetach()
    c.upload(_scene_frame(0)[:2000])
    assert c.size() == 2000


# ---------------------------------------------------------------- single-process multi-device mode (pft_tracker_set_devices)
def _multi_device_tracker(kld, devices, parity=False):
    from pcl_tracking_b200 import pcl
    from tests import util
    ctx = pcl.Context(devices[0])
    scene, model, centre = util.small_case(77, n_scene=4000, n_model=260)
    g = (pcl.KLDAdaptiveParticleFilterOMPTracker if kld else pcl.ParticleFilterOMPTracker)(16, ctx=ctx)
    g.setDevices(devices)  # first call on the new tracker: the setters below reach every device
    pcl.configure_like_reference(g, coherence_cls=lambda: _coherence(parity), particle_num=N_PART, max_particle_num=N_MAX,
                                 use_hsv=True, iteration_num=2)
    if kld:
        g.setEpsilon(0.2)
        g.setBinSize([0.1] * 6)
    m = np.eye(4, dtype=np.float32)
    m[:3, 3] = centre
    g.setTrans(m)
    g.seed(99)
    g.setReferenceCloud(model)
    cloud = pcl.PointCloud(scene, ctx=ctx)
    g.setInputCloud(cloud)
    return ctx, g, cloud


@pytest.mark.parametrize("kld,n_dev,parity", [(False, 2, False), (True, 3, False), (False, 2, True)], ids=["False-2", "True-3", "parity-False-2"])
def test_one_tracker_object_drives_several_devices(kld, n_dev, parity):
    """One process, one tracker object, n ranks: bit-identical to the plain single-GPU tracker over several frames (graph
    replays included), with the exact search and with the parity search.  With fewer GPUs than ranks the ranks share
    GPU 0 (two contexts of this process on one device)."""
    import torch
    have = torch.cuda.device_count()
    devices = list(range(n_dev)) if have >= n_dev else [0] * n_dev
    ctx, g, cloud = _multi_device_tracker(kld, devices, parity)
    got = _run(g)
    assert g.graphReplays() >= 1
    ctx1, g1, cloud1 = _tracker(kld, parity=parity)
    want = _run(g1)
    for f in range(FRAMES):
        for j, name in enumerate(("particles", "raw weights", "result")):
            assert np.array_equal(got[f][j].view(np.uint32), want[f][j].view(np.uint32)), "%s differ: frame %d" % (name, f)
    # the library-owned trackers of the other ranks hold the same replicated state
    for r in range(1, n_dev):
        fr = g.follower(r)
        assert np.array_equal(fr.getParticles().view(np.uint32), want[-1][0].view(np.uint32)), "rank %d differs" % r
        assert np.array_equal(fr.rawWeights().view(np.uint32), want[-1][1].view(np.uint32)), "rank %d differs" % r


def test_set_devices_must_come_first():
    from pcl_tracking_b200 import pcl
    ctx, g, cloud = _tracker(False)
    g.compute()
    with pytest.raises(pcl.PftError):
        g.setDevices([0, 0])


def test_weight_phase_refuses_a_peer_attached_tracker():
    """The phase API leaves the exchanges to its caller, so a tracker whose kernels exchange through peer windows refuses
    it: a host check, before anything is launched."""
    from pcl_tracking_b200 import pcl
    ctx, g, cloud = _multi_device_tracker(False, [0, 0])
    g.compute()
    with pytest.raises(pcl.PftError):
        g.weightPhase(0)
