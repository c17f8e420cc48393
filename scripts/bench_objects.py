"""One object per GPU: frames/s of the multi-object workloads with the trackers placed over 1, 2, 4 and 8 devices.

Workloads (the scene is downsampled on device 0 every frame; L2 is flushed on every device between steps):
  c5   8 objects x 1000 particles (fixed N) in the 217 088-point scene;
  qhd  the reference's literal configuration with 8 objects: KLD 400 / <= 500 particles, 518 400-point frames.
Object k runs on device k % d, on the sensor's own context for device 0 and on one context per further device, which
reads the scene through its replica (pft_tracker_set_input_cloud with a cloud of another context).  Every placement runs
in the reference's serial loop (setInputCloud + compute per tracker) and through pft_compute_batch, the placements in
alternating order.  A step is timed with CUDA events on the sensor's stream, after every context stream has joined it.
The fan-out (the copy of the downsampled scene into the replicas) is timed apart, in a run of its own with host
synchronisation between steps: events on the sensor's stream around the one fan-out launch of a pft_compute_batch
whose trackers all sit on other contexts.  The poses of every placement must equal the 1-device poses.

usage: python scripts/bench_objects.py [--steps 60] [--warmup 5] [--reps 2] [--workloads c5,qhd] [--out FILE]
Prints one JSON line.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import bench  # noqa: E402  (frame and model helpers)

N_OBJECTS = 8


def gpu_info(n):
    """Name and power limit of the first n devices, read in the same run as the measurement."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout
        rows = [[c.strip() for c in l.split(",")] for l in out.strip().splitlines()]
        return [{"index": int(r[0]), "name": r[1], "power_limit": r[2]} for r in rows[:n]]
    except Exception as e:  # pragma: no cover
        return [{"error": repr(e)}]


def workload_frames(workload):
    from pcl_tracking_b200 import synth
    if workload == "c5":
        return bench.make_frames(bench.N_FRAMES, N_OBJECTS)
    objs = synth.default_objects(N_OBJECTS, seed=3)
    frames, oid0 = [], None
    for f in range(bench.N_FRAMES):
        pts, oid = synth.render(f, objs, sensor=synth.KINECT2_QHD)
        oid0 = oid if f == 0 else oid0
        frames.append(pts)
    return frames, oid0


class Placement:
    """The 8 trackers of one workload with object k on device k % n_dev (device 0: the sensor's context)."""

    def __init__(self, pcl, workload, sensor, ctxs, models, batch, torch):
        self.pcl, self.sensor, self.batch, self.torch = pcl, sensor, batch, torch
        self.ctxs = ctxs
        self.trackers = []
        for k, (model, centroid) in enumerate(models):
            ctx = ctxs[k % len(ctxs)]
            if workload == "qhd":
                t = pcl.KLDAdaptiveParticleFilterOMPTracker(16, ctx=ctx)
                pcl.configure_like_reference(t, particle_num=400, max_particle_num=500, use_hsv=True, iteration_num=bench.ITERATIONS)
            else:
                t = pcl.ParticleFilterOMPTracker(16, ctx=ctx)
                pcl.configure_like_reference(t, particle_num=bench.PARTICLES_PER_GPU, use_hsv=True, iteration_num=bench.ITERATIONS)
            m = np.eye(4, dtype=np.float32)
            m[:3, 3] = centroid
            t.setTrans(m)
            t.seed(1234 + k)
            t.setReferenceCloud(model)
            self.trackers.append(t)
        self.streams = [torch.cuda.ExternalStream(c.stream, device="cuda:%d" % c.device) for c in ctxs]
        self.k = 0

    def step(self):
        ds = self.sensor.frame(bench.frame_order(self.k, bench.N_FRAMES))
        for t in self.trackers:
            t.setInputCloud(ds)
        if self.batch:
            self.pcl.compute_batch(self.trackers)
        else:
            for t in self.trackers:
                t.compute()
        self.k += 1

    def join(self):
        """The sensor's stream waits for every context stream."""
        for s in self.streams[1:]:
            ev = self.torch.cuda.Event()
            ev.record(s)
            self.streams[0].wait_event(ev)

    def poses(self):
        return np.array([t.getResult().tolist() for t in self.trackers], dtype=np.float32)


class Sensor:
    def __init__(self, pcl, ctx, frames):
        self.raw = [pcl.PointCloud(f, ctx=ctx) for f in frames]
        self.ds = pcl.PointCloud(ctx=ctx)
        self.vg = pcl.ApproximateVoxelGrid(ctx=ctx)
        self.vg.setLeafSize(bench.LEAF, bench.LEAF, bench.LEAF)
        self.vg.setPassThrough("z", 0.0, 10.0)

    def frame(self, f):
        self.vg.setInputCloud(self.raw[f])
        self.vg.filter(self.ds)
        return self.ds


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--reps", type=int, default=2, help="timed passes per placement, placements in alternating order")
    ap.add_argument("--workloads", default="c5,qhd")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if args.steps < 1 or args.reps < 1:
        ap.error("--steps and --reps must be >= 1")
    import torch
    from pcl_tracking_b200 import pcl
    n_have = torch.cuda.device_count()
    if n_have < 1:
        raise SystemExit("no CUDA device: this script measures the GPU and has no CPU fallback")
    counts = [d for d in (1, 2, 4, 8) if d <= n_have]
    flush = [torch.empty(256 << 20, dtype=torch.uint8, device="cuda:%d" % d) for d in range(max(counts))]
    ctx0 = pcl.Context(0)
    dev_ctx = {0: ctx0}
    for d in range(1, max(counts)):
        dev_ctx[d] = pcl.Context(d)
    record = {"script": "scripts/bench_objects.py", "gpus": gpu_info(max(counts)), "steps": args.steps, "warmup": args.warmup, "reps": args.reps,
              "l2": "flushed on every device between timed steps (256 MiB write each)", "objects": N_OBJECTS, "workloads": {}}
    for workload in args.workloads.split(","):
        frames, oid0 = workload_frames(workload)
        sensor = Sensor(pcl, ctx0, frames)
        models = [pcl.prepare_model(pcl.PointCloud(bench.raw_model(frames, oid0, k), ctx=ctx0), bench.LEAF, ctx=ctx0) for k in range(N_OBJECTS)]
        sets = {}
        for d in counts:
            for batch in (False, True):
                p = Placement(pcl, workload, sensor, [dev_ctx[i] for i in range(d)], models, batch, torch)
                for _ in range(args.warmup):
                    p.step()
                sets[(d, batch)] = p
        torch.cuda.synchronize()
        ms = {key: 0.0 for key in sets}
        order = list(sets)
        for rep in range(args.reps):
            for key in (order if rep % 2 == 0 else order[::-1]):
                p = sets[key]
                ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
                for d in range(len(p.ctxs)):
                    dev_ctx[d].synchronize()
                torch.cuda.synchronize()
                for i in range(args.steps):
                    for d, s in enumerate(p.streams):
                        with torch.cuda.stream(s):
                            flush[d].fill_(1)
                    p.join()
                    ev[i][0].record(p.streams[0])
                    p.step()
                    p.join()
                    ev[i][1].record(p.streams[0])
                for d in range(len(p.ctxs)):
                    dev_ctx[d].synchronize()
                ms[key] += sum(a.elapsed_time(b) for a, b in ev)
        want = sets[(1, False)].poses()
        res = {}
        for (d, batch), p in sets.items():
            got = p.poses()
            assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), "%s: poses on %d devices (%s) differ from 1 device" % (
                workload, d, "batch" if batch else "serial loop")
            res.setdefault(str(d), {})["batch_fps" if batch else "serial_fps"] = round(1000.0 * args.steps * args.reps / ms[(d, batch)], 1)
        # fan-out time: every tracker on a context other than the sensor's (device 0 included, as a context of its own)
        fan = {}
        for d in counts:
            extra = [pcl.Context(0)] + [dev_ctx[i] for i in range(1, d)]
            p = Placement(pcl, workload, sensor, extra, models, True, torch)
            s0 = torch.cuda.ExternalStream(ctx0.stream, device="cuda:0")
            for _ in range(args.warmup):
                p.step()
            t_us, n_pts = [], 0
            for i in range(args.steps):
                for c in extra:
                    c.synchronize()
                ctx0.synchronize()
                ds = sensor.frame(bench.frame_order(p.k, bench.N_FRAMES))
                for t in p.trackers:
                    t.setInputCloud(ds)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(s0)
                pcl.compute_batch(p.trackers)  # one fan-out launch into the replicas of all `extra` contexts
                b.record(s0)
                p.k += 1
                ctx0.synchronize()
                t_us.append(1000.0 * a.elapsed_time(b))
                n_pts = ds.size()
            for c in extra:
                c.synchronize()
            fan[str(d)] = {"destinations": len(extra), "points": int(n_pts), "us_per_launch_median": round(float(np.median(t_us)), 2)}
        record["workloads"][workload] = {"frames_per_s": res, "fanout": fan, "scene_points": len(frames[0]),
                                         "poses_equal_1_device": True}
    line = json.dumps(record)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    t0 = time.time()
    main()
    print("# %.0f s" % (time.time() - t0), file=sys.stderr)
