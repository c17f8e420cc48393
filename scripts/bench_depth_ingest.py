#!/usr/bin/env python
"""Frames/s of one tracked camera frame, end to end, through the two host ingests of the library:

  pointcloud2  the sensor_msgs/PointCloud2 payload of 32-byte pcl::PointXYZRGBA records (pft_cloud_upload_pointcloud2),
               what the reference's callback receives from /kinect2/<res>/points (ref: src/auto_tracking.cpp:619-622, :775);
  images       the registered 16UC1 depth + bgr8 colour images that topic is computed from, 5 bytes per pixel
               (pft_cloud_upload_depth_image: two copies + depth_image_kernel).

A step is: upload the frame from pinned host memory, PassThrough(z in [0, 10]) + 1 cm voxel grid, compute(), read the
pose back -- as bench.py's e2e.  Both ingests run alternately, step by step, each with its own identically seeded
tracker, synchronously and double-buffered (frame k + 1 uploaded on the copy stream while frame k is tracked; two
clouds); the poses of the two ingests must be identical at every step.  L2 is flushed (256 MiB write) before every
step, outside the timed span.  Workloads as bench.py: c2 (sd, 512x424, 1000 particles) and qhd (960x540, the
reference's KLD tracker of 400 / at most 500 particles).  The conversion kernel is also timed alone (torch.profiler,
device time of depth_image_kernel per launch) and the synchronous image upload as a whole (CUDA events), for each of
the encoding pairs in ENCODINGS: 16UC1 + bgr8 (5 bytes per pixel over PCIe), 32FC1 + rgb8 (7), 32FC1 + bgra8 (8) and
16UC1 depth alone (2).

Workload `registered`: a Kinect2 whose depth is not registered to its colour camera, sd 16UC1 depth (512x424) from
the depth sensor and qhd bgr8 colour (960x540) from a camera 52 mm away, registered on the device
(pft_cloud_upload_depth_images_reg, fill_upsampling on) and converted, against the already-registered qhd 16UC1 depth +
bgr8 colour of the same scene.  It reports the H2D bytes per frame, the three register kernels' device time per frame
(torch.profiler) and the frames/s end to end with tracking (the qhd tracker), synchronous and double-buffered.  The
two arms see different clouds, so their poses are not compared.

Needs a CUDA device; prints the card's name and power limit with the numbers, one JSON line per workload.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from bench import ITERATIONS, LEAF, N_FRAMES, frame_order  # noqa: E402

# the depth + colour encodings the conversion is timed in: the Kinect2 pair, the Gazebo Kinect plugin's depth with an
# rgb8 and a bgra8 camera, and depth alone
ENCODINGS = [("16UC1", "bgr8"), ("32FC1", "rgb8"), ("32FC1", "bgra8"), ("16UC1", "none")]
BYTES_PER_PIXEL = {"16UC1": 2, "32FC1": 4, "bgr8": 3, "rgb8": 3, "bgra8": 4, "none": 0}


def encode_depth(depth_mm, encoding):
    """A uint16 millimetre image in `encoding`: as it is, or float32 metres with NaN for no return."""
    if encoding == "16UC1":
        return depth_mm
    return np.where(depth_mm == 0, np.float32(np.nan), depth_mm.astype(np.float32) * np.float32(0.001)).astype(np.float32)


def encode_colour(bgr, encoding):
    """A bgr8 image in `encoding`."""
    if encoding == "bgr8":
        return bgr
    if encoding == "rgb8":
        return np.ascontiguousarray(bgr[..., ::-1])
    return np.concatenate([bgr, np.full(bgr.shape[:2] + (1,), 255, np.uint8)], axis=2)  # bgra8


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:  # the numbers stay, the card's limit is then reported as unknown
        out = "unknown (%s)" % e
    return {"device": name, "power_limit_and_max_sm_clock": out}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200, help="timed steps per ingest and mode")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workloads", default="c2,qhd,registered")
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_depth_ingest.py: no CUDA device (the library has no CPU fallback)")
    from pcl_tracking_b200 import pcl, synth

    ctx = pcl.Context(0)
    stream = torch.cuda.ExternalStream(ctx.stream, device=torch.device("cuda", 0))
    flush_buf = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    head = card()
    lines = [dict(head, what="card")]
    print(json.dumps(lines[0]), flush=True)

    for workload in args.workloads.split(","):
        if workload == "registered":
            lines += registered_workload(args, ctx, stream, flush_buf)
            continue
        sensor = synth.KINECT2_QHD if workload == "qhd" else synth.KINECT2_SD
        w, h = sensor["width"], sensor["height"]
        objs = synth.default_objects(1)
        images, oid0 = [], None
        for f in range(N_FRAMES):
            pts, oid = synth.render(f, objs, sensor=sensor)
            oid0 = oid if f == 0 else oid0
            images.append(synth.depth_images(pts, sensor))
        K = images[0][2]
        fx, fy, cx, cy = K[0, 0], K[1, 1], K[0, 2], K[1, 2]
        # the PointCloud2 payload of each frame: the 32-byte records of the cloud the images convert to, so that both
        # ingests deliver the same points
        payloads = [pcl.PointCloud(ctx=ctx).fromDepthImage(d, c, fx, fy, cx, cy).to_numpy(pcl32=True) for d, c, _ in images]
        pin32 = [pcl.PinnedBuffer.of(p) for p in payloads]
        pin_img = [(pcl.PinnedBuffer.of(d), pcl.PinnedBuffer.of(c)) for d, c, _ in images]
        raw = pcl.PointCloud(ctx=ctx).fromDepthImage(images[0][0], images[0][1], fx, fy, cx, cy).to_numpy()
        model, centre = pcl.prepare_model(pcl.PointCloud(synth.model_points(raw, oid0, 0), ctx=ctx), LEAF, ctx=ctx)

        def tracker():
            if workload == "qhd":
                t = pcl.KLDAdaptiveParticleFilterOMPTracker(16, ctx=ctx)
                pcl.configure_like_reference(t, particle_num=400, max_particle_num=500, use_hsv=True, iteration_num=ITERATIONS)
            else:
                t = pcl.ParticleFilterOMPTracker(16, ctx=ctx)
                pcl.configure_like_reference(t, particle_num=1000, use_hsv=True, iteration_num=ITERATIONS)
            m = np.eye(4, dtype=np.float32)
            m[:3, 3] = centre
            t.setTrans(m)
            t.seed(1234)
            t.setReferenceCloud(model)
            return t

        def upload(ingest, cloud, k, asynchronous):
            f = frame_order(k, N_FRAMES)
            if ingest == "images":
                cloud.fromDepthImage(pin_img[f][0].ptr, pin_img[f][1].ptr, fx, fy, cx, cy, asynchronous=asynchronous, width=w, height=h)
            else:
                cloud.fromPointCloud2(pin32[f].ptr, w, h, 32, asynchronous=asynchronous)

        class Arm:
            def __init__(self, ingest, pipelined):
                self.ingest, self.pipelined = ingest, pipelined
                self.t, self.vg, self.ds = tracker(), pcl.ApproximateVoxelGrid(ctx=ctx), pcl.PointCloud(ctx=ctx)
                self.vg.setLeafSize(LEAF, LEAF, LEAF)
                self.vg.setPassThrough("z", 0.0, 10.0)
                self.clouds = [pcl.PointCloud(ctx=ctx), pcl.PointCloud(ctx=ctx)]
                self.ms = 0.0
                if pipelined:
                    upload(ingest, self.clouds[0], 0, True)

            def step(self, k):
                if self.pipelined:
                    upload(self.ingest, self.clouds[(k + 1) % 2], k + 1, True)
                else:
                    upload(self.ingest, self.clouds[k % 2], k, False)
                self.vg.setInputCloud(self.clouds[k % 2])
                self.vg.filter(self.ds)
                self.t.setInputCloud(self.ds)
                self.t.compute()
                return np.array(self.t.getResult()).tobytes()  # D2H of the pose: synchronises

        for pipelined in (False, True):
            arms = [Arm("pointcloud2", pipelined), Arm("images", pipelined)]
            for k in range(args.warmup + args.steps):
                poses = []
                for arm in arms:
                    with torch.cuda.stream(stream):
                        flush_buf.fill_(1)
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(stream)
                    poses.append(arm.step(k))
                    e1.record(stream)
                    e1.synchronize()
                    if k >= args.warmup:
                        arm.ms += e0.elapsed_time(e1)
                if poses[0] != poses[1]:
                    raise AssertionError("%s %s step %d: the two ingests gave different poses" % (workload, "pipelined" if pipelined else "sync", k))
            ctx.synchronize()
            rec = {"what": "e2e", "workload": workload, "width": w, "height": h, "mode": "pipelined" if pipelined else "sync",
                   "steps": args.steps, "poses_identical_every_step": True}
            for arm, nbytes in zip(arms, (32 * w * h, 5 * w * h)):
                ms = arm.ms / args.steps
                rec[arm.ingest] = {"h2d_bytes_per_step": nbytes, "ms_per_step": ms, "frames_per_s": 1e3 / ms}
            lines.append(rec)
            print(json.dumps(rec), flush=True)

        # the conversion kernel alone (device time per launch, torch.profiler) and the synchronous image upload as a
        # whole (H2D copies + kernel + header, CUDA events), L2 flushed before each, for each pair of encodings: the
        # frames' images re-encoded as a camera of that pair would publish them (32FC1: metres, NaN where 16UC1 has 0)
        from torch.profiler import ProfilerActivity, profile
        cloud = pcl.PointCloud(ctx=ctx)
        reps = 100
        for denc, cenc in ENCODINGS:
            pins = [(pcl.PinnedBuffer.of(encode_depth(d, denc)), pcl.PinnedBuffer.of(encode_colour(c, cenc)) if cenc != "none" else None)
                    for d, c, _ in images]
            up_ms = 0.0
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for k in range(reps):
                    with torch.cuda.stream(stream):
                        flush_buf.fill_(1)
                    f = frame_order(k, N_FRAMES)
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(stream)
                    cloud.fromDepthImage(pins[f][0].ptr, pins[f][1].ptr if pins[f][1] else None, fx, fy, cx, cy, width=w, height=h,
                                         depth_encoding=denc, colour_encoding=cenc)
                    e1.record(stream)
                    e1.synchronize()
                    up_ms += e0.elapsed_time(e1)
            kern = [e for e in prof.key_averages() if "depth_image_kernel" in e.key]
            kernel_us = (getattr(kern[0], "device_time_total", None) or kern[0].cuda_time_total) / kern[0].count if kern else None
            pixel = BYTES_PER_PIXEL[denc] + BYTES_PER_PIXEL[cenc]
            rec = {"what": "kernel", "workload": workload, "width": w, "height": h, "depth_encoding": denc, "colour_encoding": cenc,
                   "h2d_bytes_per_frame": pixel * w * h, "launches": kern[0].count if kern else 0, "depth_image_kernel_us": kernel_us,
                   "kernel_bytes": (pixel + 16) * w * h, "kernel_gb_per_s": ((pixel + 16) * w * h / (kernel_us * 1e-6) / 1e9) if kernel_us else None,
                   "image_upload_us": up_ms / reps * 1e3}
            lines.append(rec)
            print(json.dumps(rec), flush=True)
            for d, c in pins:
                d.free()
                if c:
                    c.free()
        for b in pin32:
            b.free()
        for d, c in pin_img:
            d.free()
            c.free()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


def registered_workload(args, ctx, stream, flush_buf):
    import torch
    from torch.profiler import ProfilerActivity, profile

    from pcl_tracking_b200 import pcl, synth
    sd, qhd = synth.KINECT2_SD, synth.KINECT2_QHD
    w, h = qhd["width"], qhd["height"]
    offset = np.array([0.052, 0.0, 0.0])  # the colour camera in the depth camera's frame
    colour_pose = (np.eye(3), offset)
    M = np.eye(4)[:3].copy()
    M[:, 3] = -offset
    objs = synth.default_objects(1)
    frames = []
    for f in range(N_FRAMES):
        depth_sd, _, Kd = synth.depth_images(synth.render(f, objs, sensor=sd)[0], sd)
        pts, oid = synth.render(f, objs, sensor=qhd, camera=colour_pose)
        depth_qhd, bgr, Kc = synth.depth_images(pts, qhd)
        frames.append((pcl.PinnedBuffer.of(depth_sd), pcl.PinnedBuffer.of(bgr), pcl.PinnedBuffer.of(depth_qhd), oid if f == 0 else None))
    fx, fy, cx, cy = Kc[0, 0], Kc[1, 1], Kc[0, 2], Kc[1, 2]
    reg = dict(depth_K=Kd, depth_to_colour=M, fill_upsampling=True, depth_width=sd["width"], depth_height=sd["height"])

    def upload(ingest, cloud, k, asynchronous):
        d_sd, bgr, d_qhd, _ = frames[frame_order(k, N_FRAMES)]
        cam = dict(bgr=bgr.ptr, width=w, height=h, fx=fx, fy=fy, cx=cx, cy=cy)
        if ingest == "register":
            cam.update(depth=d_sd.ptr, registration=reg)
        else:
            cam.update(depth=d_qhd.ptr)
        cloud.fromDepthImages([cam], asynchronous=asynchronous)

    raw = pcl.PointCloud(ctx=ctx)
    upload("registered", raw, 0, False)
    model, centre = pcl.prepare_model(pcl.PointCloud(synth.model_points(raw.to_numpy(), frames[0][3], 0), ctx=ctx), LEAF, ctx=ctx)

    def tracker():
        t = pcl.KLDAdaptiveParticleFilterOMPTracker(16, ctx=ctx)
        pcl.configure_like_reference(t, particle_num=400, max_particle_num=500, use_hsv=True, iteration_num=ITERATIONS)
        m = np.eye(4, dtype=np.float32)
        m[:3, 3] = centre
        t.setTrans(m)
        t.seed(1234)
        t.setReferenceCloud(model)
        return t

    lines = []
    bytes_per_frame = {"register": 2 * sd["width"] * sd["height"] + 3 * w * h, "registered": 5 * w * h}
    for pipelined in (False, True):
        rec = {"what": "e2e", "workload": "registered", "width": w, "height": h, "mode": "pipelined" if pipelined else "sync", "steps": args.steps}
        for ingest in ("register", "registered"):
            t, vg, ds = tracker(), pcl.ApproximateVoxelGrid(ctx=ctx), pcl.PointCloud(ctx=ctx)
            vg.setLeafSize(LEAF, LEAF, LEAF)
            vg.setPassThrough("z", 0.0, 10.0)
            clouds = [pcl.PointCloud(ctx=ctx), pcl.PointCloud(ctx=ctx)]
            if pipelined:
                upload(ingest, clouds[0], 0, True)
            ms = 0.0
            for k in range(args.warmup + args.steps):
                with torch.cuda.stream(stream):
                    flush_buf.fill_(1)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                if pipelined:
                    upload(ingest, clouds[(k + 1) % 2], k + 1, True)
                else:
                    upload(ingest, clouds[k % 2], k, False)
                vg.setInputCloud(clouds[k % 2])
                vg.filter(ds)
                t.setInputCloud(ds)
                t.compute()
                t.getResult()  # D2H of the pose: synchronises
                e1.record(stream)
                e1.synchronize()
                if k >= args.warmup:
                    ms += e0.elapsed_time(e1)
            ms /= args.steps
            rec[ingest] = {"h2d_bytes_per_step": bytes_per_frame[ingest], "ms_per_step": ms, "frames_per_s": 1e3 / ms}
        lines.append(rec)
        print(json.dumps(rec), flush=True)

    # the register kernels alone (device time per frame) and the synchronous upload as a whole, L2 flushed before each
    cloud = pcl.PointCloud(ctx=ctx)
    reps = 100
    for ingest in ("register", "registered"):
        up_ms = 0.0
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for k in range(reps):
                with torch.cuda.stream(stream):
                    flush_buf.fill_(1)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                upload(ingest, cloud, k, False)
                e1.record(stream)
                e1.synchronize()
                up_ms += e0.elapsed_time(e1)
        kernels = {}
        for e in prof.key_averages():
            for name in ("register_reset_kernel", "register_zbuffer_kernel", "register_finalise_kernel", "depth_image_kernel"):
                if name in e.key:
                    kernels[name] = (getattr(e, "device_time_total", None) or e.cuda_time_total) / reps
        rec = {"what": "kernel", "workload": "registered", "ingest": ingest, "h2d_bytes_per_frame": bytes_per_frame[ingest],
               "kernel_us_per_frame": kernels, "register_us_per_frame": sum(v for k, v in kernels.items() if k.startswith("register")),
               "image_upload_us": up_ms / reps * 1e3}
        lines.append(rec)
        print(json.dumps(rec), flush=True)
    for d_sd, bgr, d_qhd, _ in frames:
        d_sd.free()
        bgr.free()
        d_qhd.free()
    return lines


if __name__ == "__main__":
    main()
