#!/usr/bin/env python
"""Frames/s of one tracked frame fused from 1, 2 or 4 calibrated depth cameras (pft_cloud_upload_depth_images: the
images of every camera copied from pinned memory, converted and moved into the common frame by one launch of
depth_image_kernel), end to end.

A step is: upload the cameras' images, PassThrough(z in [0, 10]) + 1 cm voxel grid, compute(), read the pose back --
as bench_depth_ingest.py.  Camera 0 is the default synthetic viewpoint and its optical frame is the common frame; the
others look at the same table from other sides (synth.side_camera() and two more look_at poses).  Workloads: every
camera at sd (512x424, ParticleFilterOMPTracker, 1000 particles) or at qhd (960x540, the reference's KLD tracker of
400 / at most 500 particles), run synchronously and double-buffered (frame k + 1 uploaded on the copy stream while
frame k is tracked).  L2 is flushed (256 MiB write) before every step, outside the timed span.  At every step the pose
must equal the pose of an identically seeded tracker fed the host composition of the same frame (each camera through
fromDepthImage, downloaded, transformed as pcl::transformPointCloud does on the host, concatenated, uploaded).  The
kernel is also timed alone (torch.profiler, device time of depth_image_kernel per launch, 21 B moved per pixel).

Then one occlusion scenario, reported without any assertion: a static box stands between camera 0 and object 0 for a
stretch of frames while the side camera still sees the object.  For camera 0 alone and for the fused scene, the
distance between the tracked model's centroid (getResultBox) and its true position c_f + R_f R_0^T (m - c_0).

Needs a CUDA device; prints the card's name and power limit with the numbers, one JSON line per record.
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from bench import ITERATIONS, LEAF, N_FRAMES, frame_order  # noqa: E402
from scripts.bench_depth_ingest import card  # noqa: E402


def viewpoints(synth):
    """World-from-camera poses of the four cameras (None: the default camera, whose frame is the common frame)."""
    n = synth.table_frame()[2]
    return [None, synth.side_camera(), synth.look_at([-1.3, -0.2, 0.9], [0.0, 0.25, 1.15], n),
            synth.look_at([0.0, -0.9, 0.3], [0.0, 0.3, 1.2], n)]


def pcl_transform(pts, m):
    """pcl::transformPointCloud (PCL 1.8.0, cloud not dense) on the host: finite points only, one rounded fp32 op at a time."""
    m = np.asarray(m, dtype=np.float32)
    out = pts.copy()
    x, y, z = pts["x"], pts["y"], pts["z"]
    finite = np.isfinite(x) & np.isfinite(y) & np.isfinite(z)
    with np.errstate(invalid="ignore", over="ignore"):
        for r, k in enumerate(("x", "y", "z")):
            v = ((m[r, 0] * x + m[r, 1] * y) + m[r, 2] * z) + m[r, 3]
            out[k][finite] = v[finite]
    return out


def render_cameras(synth, f, objs, sensor, views):
    cams = []
    for view in views:
        pts = synth.render(f, objs, sensor=sensor, camera=view)[0]
        d, c, K = synth.depth_images(pts, sensor)
        cams.append(dict(depth=d, bgr=c, K=K, pose=None if view is None else synth.pose_matrix(view).astype(np.float32)))
    return cams


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200, help="timed steps per workload and mode")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--cameras", default="1,2,4")
    ap.add_argument("--sizes", default="sd,qhd")
    ap.add_argument("--occlusion-frames", type=int, default=30)
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_depth_cameras.py: no CUDA device (the library has no CPU fallback)")
    from torch.profiler import ProfilerActivity, profile

    from pcl_tracking_b200 import pcl, synth

    ctx = pcl.Context(0)
    stream = torch.cuda.ExternalStream(ctx.stream, device=torch.device("cuda", 0))
    flush_buf = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    lines = [dict(card(), what="card")]
    print(json.dumps(lines[0]), flush=True)

    def emit(rec):
        lines.append(rec)
        print(json.dumps(rec), flush=True)

    def tracker(size, model, centre, seed=1234):
        if size == "qhd":
            t = pcl.KLDAdaptiveParticleFilterOMPTracker(16, ctx=ctx)
            pcl.configure_like_reference(t, particle_num=400, max_particle_num=500, use_hsv=True, iteration_num=ITERATIONS)
        else:
            t = pcl.ParticleFilterOMPTracker(16, ctx=ctx)
            pcl.configure_like_reference(t, particle_num=1000, use_hsv=True, iteration_num=ITERATIONS)
        m = np.eye(4, dtype=np.float32)
        m[:3, 3] = centre
        t.setTrans(m)
        t.seed(seed)
        t.setReferenceCloud(model)
        return t

    def host_composition(cams):
        parts = []
        for c in cams:
            K = c["K"]
            p = pcl.PointCloud(ctx=ctx).fromDepthImage(c["depth"], c["bgr"], K[0, 0], K[1, 1], K[0, 2], K[1, 2]).to_numpy()
            parts.append(p if c["pose"] is None else pcl_transform(p, c["pose"][:3]))
        return np.concatenate(parts)

    views = viewpoints(synth)
    objs = synth.default_objects(1)
    for size in args.sizes.split(","):
        sensor = synth.KINECT2_QHD if size == "qhd" else synth.KINECT2_SD
        w, h = sensor["width"], sensor["height"]
        all_frames = [render_cameras(synth, f, objs, sensor, views) for f in range(N_FRAMES)]
        pts0, oid0 = synth.render(0, objs, sensor=sensor)
        c0 = all_frames[0][0]
        K = c0["K"]
        raw = pcl.PointCloud(ctx=ctx).fromDepthImage(c0["depth"], c0["bgr"], K[0, 0], K[1, 1], K[0, 2], K[1, 2]).to_numpy()
        model, centre = pcl.prepare_model(pcl.PointCloud(synth.model_points(raw, oid0, 0), ctx=ctx), LEAF, ctx=ctx)
        for ncam in (int(x) for x in args.cameras.split(",")):
            frames = [cams[:ncam] for cams in all_frames]
            pinned = [[(pcl.PinnedBuffer.of(c["depth"]), pcl.PinnedBuffer.of(c["bgr"])) for c in cams] for cams in frames]
            host = [pcl.PinnedBuffer.of(host_composition(cams)) for cams in frames]
            n_pts = ncam * w * h

            def fused(k):
                f = frame_order(k, N_FRAMES)
                return [dict(c, depth=b[0].ptr, bgr=b[1].ptr, width=w, height=h) for c, b in zip(frames[f], pinned[f])]

            class Arm:
                def __init__(self, ingest, pipelined):
                    self.ingest, self.pipelined = ingest, pipelined
                    self.t, self.vg, self.ds = tracker(size, model, centre), pcl.ApproximateVoxelGrid(ctx=ctx), pcl.PointCloud(ctx=ctx)
                    self.vg.setLeafSize(LEAF, LEAF, LEAF)
                    self.vg.setPassThrough("z", 0.0, 10.0)
                    self.clouds = [pcl.PointCloud(ctx=ctx), pcl.PointCloud(ctx=ctx)]
                    self.ms = 0.0
                    if pipelined:
                        self.upload(self.clouds[0], 0, True)

                def upload(self, cloud, k, asynchronous):
                    if self.ingest == "images":
                        cloud.fromDepthImages(fused(k), asynchronous=asynchronous)
                    elif asynchronous:
                        cloud.upload_raw_async(host[frame_order(k, N_FRAMES)].ptr, n_pts)
                    else:
                        cloud.upload_raw(host[frame_order(k, N_FRAMES)].ptr, n_pts)

                def step(self, k):
                    if self.pipelined:
                        self.upload(self.clouds[(k + 1) % 2], k + 1, True)
                    else:
                        self.upload(self.clouds[k % 2], k, False)
                    self.vg.setInputCloud(self.clouds[k % 2])
                    self.vg.filter(self.ds)
                    self.t.setInputCloud(self.ds)
                    self.t.compute()
                    return np.array(self.t.getResult()).tobytes()  # D2H of the pose: synchronises

            for pipelined in (False, True):
                arm, ref = Arm("images", pipelined), Arm("host_composition", pipelined)
                for k in range(args.warmup + args.steps):
                    with torch.cuda.stream(stream):
                        flush_buf.fill_(1)
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(stream)
                    pose = arm.step(k)
                    e1.record(stream)
                    e1.synchronize()
                    if k >= args.warmup:
                        arm.ms += e0.elapsed_time(e1)
                    if pose != ref.step(k):
                        raise AssertionError("%s x%d %s step %d: the fused ingest and the host composition gave different poses"
                                             % (size, ncam, "pipelined" if pipelined else "sync", k))
                ctx.synchronize()
                ms = arm.ms / args.steps
                emit({"what": "e2e", "size": size, "cameras": ncam, "width": w, "height": h, "points": n_pts,
                      "mode": "pipelined" if pipelined else "sync", "steps": args.steps, "h2d_bytes_per_frame": 5 * n_pts,
                      "ms_per_step": ms, "frames_per_s": 1e3 / ms, "poses_equal_host_composition_every_step": True})

            cloud = pcl.PointCloud(ctx=ctx)
            reps = 100
            cloud.fromDepthImages(fused(0))
            ctx.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for k in range(reps):
                    with torch.cuda.stream(stream):
                        flush_buf.fill_(1)
                    cloud.fromDepthImages(fused(k))
                ctx.synchronize()
            kern = [e for e in prof.key_averages() if "depth_image_kernel" in e.key]
            us = (getattr(kern[0], "device_time_total", None) or kern[0].cuda_time_total) / kern[0].count if kern else None
            emit({"what": "kernel", "size": size, "cameras": ncam, "points": n_pts, "launches": kern[0].count if kern else 0,
                  "depth_image_kernel_us": us, "kernel_bytes": 21 * n_pts,
                  "kernel_gb_per_s": (21 * n_pts / (us * 1e-6) / 1e9) if us else None})
            for pair in pinned:
                for d, c in pair:
                    d.free()
                    c.free()
            for b in host:
                b.free()

    # occlusion: a static box between camera 0 and object 0 for frames [a, b); the side camera still sees the object
    sensor = synth.KINECT2_QHD
    views2 = viewpoints(synth)[:2]
    R0, c0w = synth.object_pose(objs[0], 0)
    u, v, n = synth.table_frame()
    occ_c = 0.45 * c0w
    occluder = dict(kind="box", centre=occ_c, size=np.array([0.35, 0.35, 0.02]), colour=(90, 90, 90), R0=np.eye(3), vel=np.zeros(3),
                    axis=n, rate=0.0)  # a plate facing camera 0
    nf = args.occlusion_frames
    a, b = nf // 6, nf // 2
    pts0, oid0 = synth.render(0, objs, sensor=sensor)
    raw = synth.model_points(pts0, oid0, 0)
    m_pts = np.stack([raw["x"], raw["y"], raw["z"]], axis=1).astype(np.float64)
    model, centre = pcl.prepare_model(pcl.PointCloud(raw, ctx=ctx), LEAF, ctx=ctx)
    m_centroid = m_pts.mean(axis=0)
    err = {"camera0": [], "fused": []}
    seen = {"camera0": [], "fused": []}
    arms = {name: tracker("qhd", model, centre, seed=77) for name in err}
    vg, cloud, ds = pcl.ApproximateVoxelGrid(ctx=ctx), pcl.PointCloud(ctx=ctx), pcl.PointCloud(ctx=ctx)
    vg.setLeafSize(LEAF, LEAF, LEAF)
    vg.setPassThrough("z", 0.0, 10.0)
    for f in range(nf):
        scene_objs = objs + [occluder] if a <= f < b else objs
        cams = render_cameras(synth, f, scene_objs, sensor, views2)
        Rf, cf = synth.object_pose(objs[0], f)
        truth = cf + Rf @ R0.T @ (m_centroid - c0w)
        for name, t in arms.items():
            cloud.fromDepthImages(cams[:1] if name == "camera0" else cams)
            vg.setInputCloud(cloud)
            vg.filter(ds)
            t.setInputCloud(ds)
            t.compute()
            if a <= f < b:
                box = t.getResultBox()
                err[name].append(float(np.linalg.norm(np.asarray(box["centroid"], dtype=np.float64) - truth)))
        _, oid_cam0 = synth.render(f, scene_objs, sensor=sensor)
        seen["camera0"].append(int((oid_cam0 == 0).sum()))
    emit({"what": "occlusion", "size": "qhd", "frames": nf, "occluded_frames": [a, b], "occluder_centre": occ_c.tolist(),
          "object0_pixels_camera0_min_while_occluded": min(seen["camera0"][a:b]), "object0_pixels_camera0_before": seen["camera0"][0],
          "camera0": {"mean_m": float(np.mean(err["camera0"])), "max_m": float(np.max(err["camera0"]))},
          "fused": {"mean_m": float(np.mean(err["fused"])), "max_m": float(np.max(err["fused"]))}})
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
