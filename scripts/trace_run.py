"""Tuning aid: timeline of one stream-launched c2 frame on a PFT_TRACE build (globaltimer stamps, ns)."""
import ctypes as C, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import bench
from pcl_tracking_b200 import pcl, _capi
n_particles = int(sys.argv[1]) if len(sys.argv) > 1 else 1000
frames, oid0 = bench.make_frames(6)
ctx = pcl.Context(0)
model_cloud, centroid = pcl.prepare_model(pcl.PointCloud(bench.raw_model(frames, oid0), ctx=ctx), 0.01, ctx=ctx)
t = pcl.ParticleFilterOMPTracker(16, ctx=ctx)
pcl.configure_like_reference(t, particle_num=n_particles, use_hsv=True, iteration_num=1)
m = np.eye(4, dtype=np.float32); m[:3, 3] = centroid
t.setTrans(m); t.seed(1234); t.setReferenceCloud(model_cloud)
vg = pcl.ApproximateVoxelGrid(ctx=ctx); vg.setLeafSize(0.01); vg.setPassThrough("z", 0.0, 10.0)
ds = pcl.PointCloud(ctx=ctx)
dev = [pcl.PointCloud(f, ctx=ctx) for f in frames]
lib = _capi.load()
out = (C.c_ulonglong * 64)()
init = (C.c_ulonglong * 64)()
MINS = (0, 3, 7, 11)
for i in range(64):
    init[i] = 0xFFFFFFFFFFFFFFFF if i in MINS else 0
names = {0: "index_begin first CTA in", 1: "cand_octant last warp out", 2: "cand_build_far last out", 3: "weight_lists first CTA in", 4: "weight_lists last CTA in",
         5: "weight_lists last header+sync", 6: "weight_lists last staged (mbar)", 7: "weight_lists first warp done", 8: "weight_lists last warp done",
         11: "normalize first in"}
lib.pft_debug_trace(out, init)
for k in range(14):
    vg.setInputCloud(dev[bench.frame_order(k, 6)]); vg.filter(ds)
    t.setInputCloud(ds); t.compute()
    ctx.synchronize()
    lib.pft_debug_trace(out, init)
    if k >= 10:
        v = list(out)
        t0 = v[0]
        print("frame", k, "(graph replay)" if t.graphReplays() else "")
        for i in sorted(names):
            print("   %-34s %8.1f us" % (names[i], (v[i] - t0) / 1e3))
        print("   items: %d, mean %.2f us, longest %.1f us (item %d = particle %d chunk %d), > 8 us: %d, > 16 us: %d"
              % (v[17], v[16] / max(v[17], 1) / 1e3, v[12] / 1e3, v[13], v[13] // 21, v[13] % 21, v[14], v[15]))
