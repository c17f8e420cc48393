#!/usr/bin/env python
"""bench.py -- the tracker's headline benchmark (BASELINE.json: "tracker frames/s and particle x
model-point likelihood evals/s, 217k-pt scene").

A step is one tracked frame of ref: src/auto_tracking.cpp:cloud_cb (:637, :683, :688-697):
    PassThrough(z in [0,10]) + voxel-grid(1 cm) of the 512x424 scene  ->  setInputCloud  ->  compute()
with compute() = 2 x { resample, crop + index rebuild, weight, normalise, update }.

Workloads (config.workload):
  c2   BASELINE.json configs[1]: 217 088-pt Kinect2-shaped synthetic scene, ~2k-pt model, 1000
       particles PER GPU (fixed-N tracker), Distance+HSV coherence.  With N GPUs it is ONE tracker
       of 1000*N particles sharded by particle (weak scaling): every rank downsamples the frame and
       weights its own particles; the crop box and the raw weights travel between the GPUs as peer
       stores over NVLink issued by the producing kernels (--exchange peer, default) or through
       ncclAllReduce / ncclAllGather (--exchange nccl, with rank 0 downsampling and broadcasting the
       scene); resample/normalise/update run replicated.
  c4   BASELINE.json configs[3]: 100 000 particles in total, sharded over the N GPUs (strong scaling).
  c3   BASELINE.json configs[2]: KLD-adaptive tracker, at most 10 000 particles (epsilon 0.2, bins 0.1 m / rad as the reference),
       per-frame downsample + index rebuild; the particle count lives on the device, evals are counted there.
  c5   BASELINE.json configs[4]: 8 objects (8 models, 1000 particles each) tracked in one 217k-pt scene through
       pft_compute_batch (every tracker on its own stream, forked from / joined to the scene's stream).

`value`   = likelihood evals/s, whole job, inputs resident in HBM (raw frames pre-uploaded).
`e2e`     = the same through the public API with HOST buffers: every step uploads the raw frame from
            pinned host memory (3.47 MB) and reads the result pose back (32 B).
`e2e_pipelined` (N = 1, supplementary) = e2e with the ingest double-buffered: the upload of frame k+1 is issued on the
            library's copy stream (pft_cloud_upload_async) before frame k is tracked; every step still copies one frame
            in and reads one pose back.
--impl reference times the CPU restatement of the PCL-1.8.0 path (oracle/, "port": PCL itself is not
buildable here) on every host core of the box (the thread count is set explicitly: torchrun exports
OMP_NUM_THREADS=1); when the time budget forces fewer particles per step, the throughput reported is that of the
full workload (per-particle stages scaled, per-frame stages as timed; `cpu_baseline.sample` says so).
"""
import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "likelihood evals/s (particle x model-point), 217k-pt scene tracker frame"
UNIT = "evals/s"
N_FRAMES = 6          # pre-rendered frames, played ping-pong so that motion stays continuous
LEAF = 0.01
PARTICLES_PER_GPU = 1000
C4_PARTICLES = 100_000
C3_MAX_PARTICLES = 10_000
C5_OBJECTS = 8
ITERATIONS = 2


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


# ------------------------------------------------------------------ workload
def make_frames(n_frames, n_objects=1):
    from pcl_tracking_b200 import synth
    objs = synth.default_objects(n_objects) if n_objects == 1 else synth.default_objects(n_objects, seed=3)  # (seed 3: no two objects touch)
    frames = []
    oid0 = None
    for f in range(n_frames):
        pts, oid = synth.render(f, objs)
        if f == 0:
            oid0 = oid
        frames.append(pts)
    return frames, oid0


def frame_order(k, n_frames):
    """ping-pong 0,1,..,n-1,n-2,..,1,0,1,... (index of the frame shown at step k)"""
    period = 2 * (n_frames - 1)
    r = k % period
    return r if r < n_frames else period - r


def raw_model(frames, oid0, k=0):
    from pcl_tracking_b200 import synth
    return synth.model_points(frames[0], oid0, k)


# ------------------------------------------------------------------ clocks
class ClockSampler:
    """Samples SM clock + throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._nv = None

    def sample(self):
        if not self._nv:
            return
        nv = self._nv
        try:
            self.samples.append(float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
            try:
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
            except Exception:
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
            names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
                     0x80: "hw_power_brake_slowdown"}
            for bit, name in names.items():
                if r & bit:
                    self.reasons.add(name)
        except Exception:
            pass

    def _run(self):
        while not self._stop.is_set():
            self.sample()
            self._stop.wait(0.02)

    def start(self):
        self._stop.clear()
        self._thread = threading.Thread(target=self._run, daemon=True)
        self._thread.start()

    def stop(self):
        self.sample()
        self._stop.set()
        if self._thread:
            self._thread.join()

    def summary(self):
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------ reference arm / cpu baseline (oracle)
def oracle_tracker(model, centroid, n_particles, threads):
    import oracle
    t = oracle.Tracker(kld=False)
    oracle.configure_like_reference(t, particle_num=n_particles, max_particle_num=n_particles, use_hsv=True,
                                    nn_mode=oracle.NN_PCL_APPROX, iteration_num=ITERATIONS, threads=threads)
    t.set_i(oracle.SAMPLER, oracle.SAMPLER_ALIAS_PCL)
    m = np.eye(4, dtype=np.float32)
    m[:3, 3] = centroid
    t.set_trans(m[:3])
    t.set_reference(model)
    return t


def cpu_prepare_model(raw):
    """ref: src/auto_tracking.cpp:656-674 on the CPU (oracle restatement)."""
    import oracle
    r = oracle.remove_zero_points(raw)
    c = oracle.centroid(r)
    r["x"] -= c[0]
    r["y"] -= c[1]
    r["z"] -= c[2]
    return oracle.voxel_grid_pcl(r, LEAF), c


def cpu_frame(t, frame):
    """One cloud_cb on the CPU: PassThrough + ApproximateVoxelGrid (512-slot, as PCL) + compute()."""
    import oracle
    ds = oracle.approx_voxel_grid_pcl(oracle.passthrough(frame, 2, 0.0, 10.0), LEAF)
    t.set_input(ds)
    t.compute()


def run_cpu(frames, oid0, n_particles, steps, warmup, budget_s):
    """Times `steps` CPU frames after `warmup`.  The particle count is bounded so that the run fits
    `budget_s`: throughput in evals/s does not depend on it (weight() is linear in particles)."""
    import oracle
    # every host core this process may run on -- NOT omp_get_max_threads(): torchrun exports OMP_NUM_THREADS=1 to its
    # workers, which would time the CPU arm single-threaded whenever the driver launches it for N > 1
    try:
        threads = max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        threads = max(1, os.cpu_count() or 1)
    model, centroid = cpu_prepare_model(raw_model(frames, oid0))
    M = len(model)
    # calibrate on a small particle set
    cal = oracle_tracker(model, centroid, 64, threads)
    cpu_frame(cal, frames[0])
    t0 = time.perf_counter()
    cpu_frame(cal, frames[1])
    dt = time.perf_counter() - t0
    ds_t0 = time.perf_counter()
    oracle.approx_voxel_grid_pcl(oracle.passthrough(frames[0], 2, 0.0, 10.0), LEAF)
    ds_dt = time.perf_counter() - ds_t0
    per_particle = max((dt - ds_dt) / 64.0, 1e-6)
    per_step_budget = budget_s / max(steps + warmup, 1)
    n_fit = int(max(per_step_budget - ds_dt, 0.0) / per_particle)
    n_used = int(min(n_particles, max(n_fit, 32)))
    t = oracle_tracker(model, centroid, n_used, threads)
    for k in range(warmup):
        cpu_frame(t, frames[frame_order(k, len(frames))])
    t.stage_seconds(reset=True)
    t0 = time.perf_counter()
    for k in range(steps):
        cpu_frame(t, frames[frame_order(warmup + k, len(frames))])
    total = time.perf_counter() - t0
    stages = t.stage_seconds()
    evals = float(n_used) * M * ITERATIONS * steps
    measured = evals / total
    note = ""
    if n_used < n_particles:
        # A bounded sample must not deflate the CPU arm: the downsample, the crop and the octree rebuild cost the same
        # per frame whatever the particle count.  The throughput reported for the sample is therefore the one of the
        # FULL workload, with the per-particle stages (timed inside the oracle) scaled up and the rest kept.
        prop = min(sum(stages[k] for k in ("transform", "coherence", "normalize", "resample", "update")), total)
        full_total = (total - prop) + prop * (float(n_particles) / n_used)
        evals_per_s = float(n_particles) * M * ITERATIONS * steps / full_total
        note = "; value = full-workload throughput extrapolated from the sample (per-particle stages x %.1f, per-frame stages as timed; measured on the sample itself: %.3g evals/s)" % (float(n_particles) / n_used, measured)
    else:
        evals_per_s = measured
    return {
        "evals_per_s": evals_per_s, "frames_per_s": steps / total, "ms_per_step": 1e3 * total / steps, "cores": threads,
        "particles_used": n_used, "model_points": M, "steps": steps,
        "sample": "%d frames of the c2 workload with %d of %d particles (weight() is linear in particles), %d-pt model, "
                  "PassThrough + 512-slot ApproximateVoxelGrid + octree approxNearestSearch, %d OpenMP threads%s"
                  % (steps, n_used, n_particles, M, threads, note),
        "stage_s": {k: round(v, 4) for k, v in stages.items()},
    }


def run_cpu_c1(steps, warmup, budget_s):
    """BASELINE configs[0] on the CPU: unorganised 100 000-pt scene, 5 000-pt model, 400 particles, Distance coherence only, the oracle in
    its PCL-faithful configuration on every host core."""
    import oracle
    from pcl_tracking_b200 import synth
    try:
        threads = max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        threads = max(1, os.cpu_count() or 1)
    scene, model_raw, centre = synth.uniform_surface_scene(100_000, 5_000)
    model = oracle.voxel_grid_pcl(model_raw, LEAF)  # (already centred on its centroid)
    t = oracle.Tracker(kld=False)
    oracle.configure_like_reference(t, particle_num=400, max_particle_num=400, use_hsv=False, nn_mode=oracle.NN_PCL_APPROX, iteration_num=ITERATIONS, threads=threads)
    t.set_i(oracle.SAMPLER, oracle.SAMPLER_ALIAS_PCL)
    m = np.eye(4, dtype=np.float32)
    m[:3, 3] = centre
    t.set_trans(m[:3])
    t.set_reference(model)
    M = len(model)
    for _ in range(warmup):
        cpu_frame(t, scene)
    t.stage_seconds(reset=True)
    t0 = time.perf_counter()
    done = 0
    for _ in range(steps):
        cpu_frame(t, scene)
        done += 1
        if time.perf_counter() - t0 > budget_s:
            break
    total = time.perf_counter() - t0
    stages = t.stage_seconds()
    return {"evals_per_s": 400.0 * M * ITERATIONS * done / total, "frames_per_s": done / total, "ms_per_step": 1e3 * total / done, "cores": threads,
            "particles_used": 400, "model_points": M, "steps": done,
            "sample": "%d frames of the c1 workload (100000-pt scene, %d-pt model after the 1 cm voxel grid, 400 particles, Distance coherence), PassThrough + "
                      "512-slot ApproximateVoxelGrid + octree approxNearestSearch, %d OpenMP threads" % (done, M, threads),
            "stage_s": {k: round(v, 4) for k, v in stages.items()}}


def reference_arm(args):
    rank = env_int("RANK", 0)
    if rank != 0:
        return 0
    if args.workload == "c1":
        n_particles = 400
        r = run_cpu_c1(args.steps, args.warmup, budget_s=150.0)
    else:
        frames, oid0 = make_frames(N_FRAMES)
        n_particles = C4_PARTICLES if args.workload == "c4" else PARTICLES_PER_GPU * args.gpus
        r = run_cpu(frames, oid0, n_particles, args.steps, args.warmup, budget_s=150.0)
    wl = args.workload if args.workload in ("c1", "c4") else "c2"
    line = {
        "impl": "reference", "metric": METRIC, "value": r["evals_per_s"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "strong" if args.workload == "c4" else "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, wl, r["model_points"], n_particles, 100000 if wl == "c1" else 217088),
        "frames_per_s": r["frames_per_s"],
        "cpu_baseline": {"value": r["evals_per_s"], "unit": UNIT, "cores": r["cores"], "kind": "port", "sample": r["sample"],
                         "stage_s": r["stage_s"]},
        "e2e": {"value": r["evals_per_s"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------ our arm
def source_hash():
    """Hash of the CUDA sources the loaded libpft.so was built from: profiles/*_kernel_metrics.json carry the hash of the
    build they were captured on, and their DRAM traffic is only reported when it matches (never a stale figure)."""
    import hashlib
    h = hashlib.sha256()
    d = os.path.join(ROOT, "pcl_tracking_b200", "csrc")
    for f in sorted(os.listdir(d)):
        if f.endswith((".cu", ".cuh", ".h")):
            h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


SENSORS = {"sd": (512, 424), "qhd": (960, 540)}


class Rig:
    """What every workload of one bench process shares: context, stream, distributed state, L2 flush buffer."""

    def __init__(self, args, torch, dist, ctx, stream, rank, world, local_rank, uid):
        self.args, self.torch, self.dist, self.ctx, self.stream = args, torch, dist, ctx, stream
        self.devices = [int(d) for d in args.devices.split(",")] if getattr(args, "devices", None) else None
        self.rank, self.world, self.local_rank, self.uid = rank, world, local_rank, uid
        self.flush_buf = None if args.no_flush else torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
        self._frames = {}

    def frames(self, n_objects=1, sensor="sd"):
        key = (n_objects, sensor)
        if key not in self._frames:
            from pcl_tracking_b200 import synth
            if sensor == "sd":
                self._frames[key] = make_frames(N_FRAMES, n_objects)
            else:
                objs = synth.default_objects(1)
                fr, oid0 = [], None
                for f in range(N_FRAMES):
                    pts, oid = synth.render(f, objs, sensor=synth.KINECT2_QHD)
                    oid0 = oid if f == 0 else oid0
                    fr.append(pts)
                self._frames[key] = (fr, oid0)
        return self._frames[key]

    def flush_l2(self):
        if self.flush_buf is not None:
            with self.torch.cuda.stream(self.stream):
                self.flush_buf.fill_(1)

    def sync_all(self):
        self.ctx.synchronize()
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def timed(self, step_fn, steps, first_k, sampler=None):
        """EXACTLY `steps` steps, each bracketed by CUDA events on the library's stream; L2 flushed between
        steps outside the event pairs.  Returns (sum of step times in ms, max over ranks; wall seconds)."""
        torch = self.torch
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        self.sync_all()
        if sampler:
            sampler.start()
        wall0 = time.perf_counter()
        for i in range(steps):
            self.flush_l2()
            ev[i][0].record(self.stream)
            step_fn(first_k + i)
            ev[i][1].record(self.stream)
        self.sync_all()
        wall = time.perf_counter() - wall0
        if sampler:
            sampler.stop()
        total_ms = float(sum(a.elapsed_time(b) for a, b in ev))
        if self.world > 1:
            tt = torch.tensor([total_ms], dtype=torch.float64, device="cuda")
            self.dist.all_reduce(tt, op=self.dist.ReduceOp.MAX)
            total_ms = float(tt.item())
        return total_ms, wall


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, ds, trackers):
    """What a caller of the timed path holds after its last step, as float32 .npy files in `out_dir`:
    downsampled_cloud (N x 7: x, y, z and the r, g, b, a bytes of rgba), result (one pose per tracker) and
    particles (every tracker's particles, tracker after tracker); poses and particles carry the fields of
    pcl.PARTICLE in order (x, y, z, one, roll, pitch, yaw, weight)."""
    from numpy.lib import recfunctions as rfn
    from pcl_tracking_b200 import pcl
    pts = ds.to_numpy()
    argb = np.ascontiguousarray(pts["rgba"]).view(np.uint8).reshape(-1, 4)  # little-endian bytes of a<<24 | r<<16 | g<<8 | b
    arrays = {
        "downsampled_cloud": np.column_stack([pts["x"], pts["y"], pts["z"], argb[:, [2, 1, 0, 3]].astype(np.float32)]),
        "result": rfn.structured_to_unstructured(np.array([t.getResult() for t in trackers], dtype=pcl.PARTICLE)),
        "particles": rfn.structured_to_unstructured(np.concatenate([t.getParticles() for t in trackers])),
    }
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError("--dump-outputs: %d bytes exceed the %d-byte limit" % (total, DUMP_LIMIT_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float32))


def run_workload(rig, workload, steps, warmup, with_pipelined=True, dump_dir=None):
    """One workload on the rig's GPUs: returns the fields of its bench record (rank 0; None elsewhere).  With `dump_dir`,
    rank 0 writes the outputs of the last timed step there (dump_outputs)."""
    from pcl_tracking_b200 import pcl, synth
    args, ctx, world, rank, dist = rig.args, rig.ctx, rig.world, rig.rank, rig.dist
    sensor = "qhd" if workload == "qhd" else "sd"
    width, height = SENSORS[sensor]
    n_objects = C5_OBJECTS if workload == "c5" else 1
    frames, oid0 = rig.frames(n_objects, sensor)
    n_pts = len(frames[0])
    n_particles = {"c2": PARTICLES_PER_GPU * world * (len(rig.devices) if rig.devices else 1), "c4": C4_PARTICLES, "c3": C3_MAX_PARTICLES, "c5": PARTICLES_PER_GPU, "qhd": 400}[workload]
    scene_mode = args.scene or ("peer" if args.exchange == "peer" else "broadcast")
    owns_frames = rank == 0 or scene_mode == "replicate"

    trackers, M = [], 0
    cluster_src = None
    if n_objects > 1:
        # model acquisition on the GPU (ref: src/create_model.cpp:148-230) -- init-time, untimed: Euclidean clustering of the
        # points left after the table plane is cut away gives one model cloud per object
        keep = (oid0 >= 0) & np.isfinite(frames[0]["x"])
        cluster_src = pcl.PointCloud(frames[0][keep], ctx=ctx)
        ec = pcl.EuclideanClusterExtraction(ctx=ctx)
        ec.setClusterTolerance(0.02)
        ec.setMinClusterSize(200)
        ec.setMaxClusterSize(25000)
        ec.setInputCloud(cluster_src)
        if len(ec.extract()) != n_objects:
            raise RuntimeError("expected %d clusters, got %d" % (n_objects, len(ec.sizes)))
    for k in range(n_objects):
        # model preparation on the GPU (ref :656-674) -- init-time, untimed
        raw_model_cloud = ec.cluster_cloud(k) if cluster_src is not None else pcl.PointCloud(raw_model(frames, oid0, k), ctx=ctx)
        model_cloud, centroid = pcl.prepare_model(raw_model_cloud, LEAF, ctx=ctx)
        M += model_cloud.size()
        if workload in ("c3", "qhd"):
            tracker = pcl.KLDAdaptiveParticleFilterOMPTracker(16, ctx=ctx, devices=rig.devices)
            if workload == "c3":
                pcl.configure_like_reference(tracker, particle_num=n_particles, max_particle_num=n_particles, use_hsv=True, iteration_num=ITERATIONS)
                tracker.setEpsilon(args.kld_epsilon)
                tracker.setBinSize([args.kld_bin] * 6)
            else:  # the reference's literal configuration (ref: src/auto_tracking.cpp:211-231, :775)
                pcl.configure_like_reference(tracker, particle_num=400, max_particle_num=500, use_hsv=True, iteration_num=ITERATIONS)
        else:
            tracker = pcl.ParticleFilterOMPTracker(16, ctx=ctx, devices=rig.devices)
            pcl.configure_like_reference(tracker, particle_num=n_particles, use_hsv=True, iteration_num=ITERATIONS)
        m = np.eye(4, dtype=np.float32)
        m[:3, 3] = centroid
        tracker.setTrans(m)
        tracker.seed(1234 + k)
        if world > 1 and args.exchange == "nccl":
            tracker.commInit(world, rank, rig.uid)
        elif world > 1:
            # NVLink peer exchange: windows mapped with CUDA IPC, handles shipped by torch.distributed
            tracker.setShard(world, rank)
            handles = [None] * world
            dist.all_gather_object(handles, tracker.peerExport())
            tracker.peerAttach(handles)
            dist.barrier()
        tracker.setReferenceCloud(model_cloud)
        trackers.append(tracker)
    tracker = trackers[0]

    def compute_all():
        if len(trackers) > 1:
            pcl.compute_batch(trackers)
        else:
            tracker.compute()

    def eval_count():
        return sum(t.evalCount() for t in trackers)

    # resident inputs: raw frames in HBM (rank 0 owns the sensor; the other ranks receive the downsampled scene)
    dev_frames = [pcl.PointCloud(f, ctx=ctx) for f in frames] if owns_frames else None
    # host inputs for e2e: what the reference's callback receives (ref: src/auto_tracking.cpp:597, :619-622) -- the payload of a
    # sensor_msgs/PointCloud2 of 32-byte pcl::PointXYZRGBA records, in pinned memory; plus the packed 16-byte layout (supplementary)
    lib = pcl.capi.load()
    pinned32, pinned16 = [], []
    if owns_frames:
        for f in frames:
            f32 = synth.to_pcl32(f)
            for arr, store in ((f32, pinned32), (f, pinned16)):
                p = C.c_void_p()
                pcl.check(lib.pft_host_alloc(C.byref(p), arr.nbytes))
                C.memmove(p, arr.ctypes.data, arr.nbytes)
                store.append(p)
    bytes32, bytes16 = int(frames[0].nbytes) * 2, int(frames[0].nbytes)
    upload_cloud = pcl.PointCloud(ctx=ctx)
    ds = pcl.PointCloud(ctx=ctx)
    vg = pcl.ApproximateVoxelGrid(ctx=ctx)
    vg.setLeafSize(LEAF, LEAF, LEAF)
    vg.setPassThrough("z", 0.0, 10.0)

    if world > 1 and scene_mode == "peer":
        # the downsampled scene of every rank is mapped by rank 0 (CUDA IPC handles shipped by torch.distributed)
        handles = [None] * world
        dist.all_gather_object(handles, ds.peerExport(n_pts))
        ds.peerAttach(handles, rank)
        dist.barrier()

    def track(cloud):
        if owns_frames:
            vg.setInputCloud(cloud)
            vg.filter(ds)
        if world > 1 and scene_mode == "broadcast":
            ds.broadcast(n_pts, 0)
        elif world > 1 and scene_mode == "peer":
            ds.peerBroadcast(0)
        for t in trackers:
            t.setInputCloud(ds)
        compute_all()

    def step_resident(k):
        track(dev_frames[frame_order(k, N_FRAMES)] if owns_frames else None)

    def step_e2e(k):  # PointCloud2 payload (32-byte records) from pinned host memory in, pose out
        if owns_frames:
            upload_cloud.fromPointCloud2(pinned32[frame_order(k, N_FRAMES)].value, width, height, 32)
        track(upload_cloud)
        return [t.getResult() for t in trackers]  # D2H of the pose(s): synchronises

    def step_e2e16(k):  # the same with the frame already packed to 16-byte points on the host
        if owns_frames:
            upload_cloud.upload_raw(pinned16[frame_order(k, N_FRAMES)].value, n_pts)
        track(upload_cloud)
        return [t.getResult() for t in trackers]

    # the same with the ingest double-buffered (SURVEY 8 f-1): frame k+1 is copied on the library's copy stream while
    # frame k is tracked; every step still copies one frame in and reads one pose back
    upload_pair = [pcl.PointCloud(ctx=ctx), pcl.PointCloud(ctx=ctx)]

    def prime_pipelined(k):
        upload_pair[k % 2].fromPointCloud2(pinned32[frame_order(k, N_FRAMES)].value, width, height, 32, asynchronous=True)

    def step_e2e_pipelined(k):
        prime_pipelined(k + 1)
        track(upload_pair[k % 2])
        return [t.getResult() for t in trackers]

    if rank == 0:
        print("bench[%s]: model %d pts, particles %d, world %d" % (workload, M, n_particles, world), file=sys.stderr)
    # ---- warm-up (builds the CUDA graph; one state read-back in the middle tells the host which kernels the steady-state
    # frame needs, so the graph of the timed region is the final one), then the timed region
    W = max(warmup, 3)
    for k in range(W):
        step_resident(k)
        if k == 0:
            for t in trackers:
                t.getResult()
    rig.sync_all()
    sampler = ClockSampler(rig.local_rank)
    launches0 = pcl.kernel_launch_count()
    evals0 = eval_count()  # counted on the device (the live particle count of a KLD tracker never travels to the host)
    total_ms, wall_s = rig.timed(step_resident, steps, W, sampler)
    evals_timed = eval_count() - evals0
    launches = pcl.kernel_launch_count() - launches0
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, ds, trackers)  # before the e2e passes below track further frames
    ms_per_step = total_ms / steps
    evals_per_step = float(evals_timed) / steps
    value = evals_per_step / (ms_per_step * 1e-3)
    graph_replays = tracker.graphReplays()

    def timed_e2e(fn, first_k, prime=None):
        if prime:
            prime(first_k)
        for k in range(3):
            fn(first_k + k)
        e0 = eval_count()
        ms, _ = rig.timed(fn, steps, first_k + 3)
        return float(eval_count() - e0) / steps / (ms / steps * 1e-3), ms / steps

    e2e_value, e2e_ms = timed_e2e(step_e2e, W + steps)
    e2e16_value, e2e16_ms = timed_e2e(step_e2e16, W + 2 * steps + 3)
    n_up = world if scene_mode == "replicate" else 1
    d2h = (32 + 64) * len(trackers)
    e2e = {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": bytes32 * n_up, "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms, "frames_per_s": 1e3 / e2e_ms,
           "ingest": "sensor_msgs/PointCloud2 payload of 32-byte pcl::PointXYZRGBA records (pft_cloud_upload_pointcloud2: H2D copy + unpack kernel), as the "
                     "reference's callback receives it (ref: src/auto_tracking.cpp:619-622)"}
    e2e16 = {"value": e2e16_value, "unit": UNIT, "h2d_bytes_per_step": bytes16 * n_up, "d2h_bytes_per_step": d2h, "ms_per_step": e2e16_ms,
             "frames_per_s": 1e3 / e2e16_ms, "ingest": "frame already packed to 16-byte {x,y,z,rgba} points on the host (pft_cloud_upload)"}
    e2e_pipe = None
    if world == 1 and owns_frames and with_pipelined:
        pv, pms = timed_e2e(step_e2e_pipelined, W + 3 * steps + 6, prime_pipelined)
        e2e_pipe = {"value": pv, "unit": UNIT, "ms_per_step": pms, "frames_per_s": 1e3 / pms, "h2d_bytes_per_step": bytes32, "d2h_bytes_per_step": d2h,
                    "how": "as e2e, with the upload of frame k+1 (pft_cloud_upload_pointcloud2_async, copy stream) issued before frame k is tracked"}

    # ---- roofline of the dominant kernel: CUDA events around every launch of it on the library's stream (the
    # kernel that evaluates the candidate lists, weight_lists_kernel; weight_kernel when the lists are off), over more
    # frames driven through the same code path without the graph
    for t in trackers:
        t.enableTiming(True)
    w_ms, n_w, c_ms = 0.0, 0, 0.0
    rsteps = min(steps, 100)
    evals0 = eval_count()
    for k in range(rsteps):
        rig.flush_l2()
        step_resident(W + k)
        for t in trackers:
            a, b = t.timing()
            w_ms += a
            c_ms += b
            n_w += ITERATIONS
    evals_per_launch = float(eval_count() - evals0) / max(n_w, 1) / (world * (len(rig.devices) if rig.devices else 1))  # this rank's share of every weight()
    for t in trackers:
        t.enableTiming(False)
    info = tracker.indexInfo()
    M_mean = float(M) / len(trackers)
    n_local = evals_per_launch / M_mean
    bytes_per_launch = 32.0 * evals_per_launch + 36.0 * n_local + 16.0 * info["n_cropped"]
    w_ms_per_launch = w_ms / max(n_w, 1)
    achieved = bytes_per_launch / (w_ms_per_launch * 1e-3) / 1e9
    peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    try:
        mp = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        peak, peak_src = float(mp["hbm_gbs"]), "measured (MEASURED_PEAKS.json, burst copy)"
    except Exception:
        pass
    kernel = "weight_lists_kernel" if info["use_lists"] else "weight_lists_kernel(row-table path: lists off for this crop)"
    # DRAM traffic of that kernel per launch: from the committed `ncu --set full` capture of this workload, and only when the
    # capture was taken on the very sources this library was built from (a stale figure is never reported)
    traffic, traffic_src = None, None
    try:
        km = json.load(open(os.path.join(ROOT, "profiles", "r02_kernel_metrics_%s.json" % workload)))
        if km.get("_source_hash") == source_hash() and world == 1:
            wk = [v for k, v in km.items() if k.startswith("weight_lists_kernel")][0]
            scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
            traffic = 0.0
            for key, val in wk.items():
                if key.startswith("dram__bytes_read.sum") or key.startswith("dram__bytes_write.sum"):
                    traffic += float(val) * scale[key.split("[")[1].rstrip("]")]
            traffic_src = "profiles/r02_kernel_metrics_%s.json (dram__bytes_read.sum + dram__bytes_write.sum of one launch, ncu --set full, same sources)" % workload
        else:
            traffic_src = "no ncu capture of these sources committed (profiles/r02_kernel_metrics_%s.json is of another build): not reported" % workload
    except Exception:
        traffic_src = "no ncu capture committed for this workload"
    result = tracker.getResult()
    if rank != 0:
        return None
    rec = {
        "value": value, "unit": UNIT, "ms_per_step": ms_per_step, "frames_per_s": 1e3 / ms_per_step, "evals_per_step": evals_per_step, "steps": steps, "warmup": W,
        "scaling": "strong" if workload == "c4" else "weak",
        "config": workload_config(args, workload, M, n_particles, n_pts, scene_mode),
        "e2e": e2e, "e2e_packed16": e2e16, "e2e_pipelined": e2e_pipe,
        "gpu_launches": int(launches), "graph_replays": int(graph_replays), "clocks": sampler.summary(),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
                     "kernel": kernel + "<HSV>", "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": bytes_per_launch, "ms_per_launch": w_ms_per_launch,
                     "evals_per_s_in_kernel": evals_per_launch / (w_ms_per_launch * 1e-3),
                     "particles_per_launch": n_local,
                     "share_of_compute": w_ms / c_ms if c_ms > 0 else None,
                     "how": "CUDA events around each %s launch on the library stream, %d frames, stream-launched (no graph); bytes = 32 x evals + 36 x particles + "
                            "16 x cropped scene points (SURVEY 8d)" % (kernel, rsteps)},
        "scene_index": info,
        "result_pose": {k: float(result[k]) for k in ("x", "y", "z", "roll", "pitch", "yaw")},
        "wall_s_timed_region": wall_s,
    }
    for store in (pinned32, pinned16):
        for p in store:
            lib.pft_host_free(p)
    return rec


def workload_config(args, workload, M, n_particles, n_pts=217088, scene_mode="replicate"):
    names = {
        "c1": "c1: BASELINE.json configs[0], unorganised 100000-pt synthetic scene, %d-pt model, %d particles, Distance coherence (CPU)" % (M, n_particles),
        "c2": "c2: BASELINE.json configs[1], 512x424 (217088-pt) Kinect2-shaped synthetic scene, %d-pt model, %d particles"
              " per GPU (one tracker sharded by particle), Distance+HSV coherence, 2 iterations/frame" % (M, PARTICLES_PER_GPU),
        "c4": "c4: BASELINE.json configs[3], 100000 particles sharded over the GPUs, 217088-pt scene, %d-pt model, Distance+HSV" % M,
        "c3": "c3: BASELINE.json configs[2], KLD-adaptive particle count (<= %d, epsilon %g, bins %g m / rad), 217088-pt scene, %d-pt model,"
              " per-frame voxel-grid downsample + index rebuild, Distance+HSV" % (C3_MAX_PARTICLES, args.kld_epsilon, args.kld_bin, M),
        "c5": "c5: BASELINE.json configs[4], %d objects (%d model points in total, %d particles each) tracked simultaneously in one 217088-pt scene"
              " (models = Euclidean clusters of the object points, pft_euclidean_clusters; pft_compute_batch), Distance+HSV" % (C5_OBJECTS, M, PARTICLES_PER_GPU),
        "qhd": "qhd: the reference's literal configuration (ref: src/auto_tracking.cpp:775, :211, :231): 960x540 (518400-pt) Kinect2 qhd-shaped synthetic scene,"
               " KLD tracker 400 particles / at most 500, epsilon 0.2, bins 0.1, %d-pt model, Distance+HSV" % M,
    }
    return {
        "workload": names[workload],
        "scene_points": n_pts, "model_points": M, "particles_total": n_particles, "iterations_per_frame": ITERATIONS,
        "leaf_m": LEAF, "max_distance_m": 0.1, "l2": "flushed between timed steps (256 MiB write)", "parallelism": ("particle-shard x%d, ONE process driving devices %s (pft_tracker_set_devices: windows mapped directly, scene by peer copy)"
                                                                                               % (len(args.devices.split(",")), args.devices)) if getattr(args, "devices", None) else
                       "particle-shard x%d" % args.gpus + ("" if args.gpus == 1 else ", %s exchange, scene %s" % (args.exchange, scene_mode)),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300, help="timed steps of the headline workload and of each e2e variant (the --also workloads "
                                                           "time min(steps, 60), c4 min(steps, 30), at least 3)")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps of the headline workload, write what its last step computed to DIR/*.npy (float32): "
                         "downsampled_cloud, result, particles; the inputs are seeded, so runs with the same arguments compare output for output")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=["c1", "c2", "c3", "c4", "c5", "qhd"])
    ap.add_argument("--also", default=None, help="comma-separated extra workloads reported under `workloads` of the same line "
                                                 "(default: c4,c3,c5,qhd on one GPU, c4 on several; 'none' for the headline workload alone)")
    ap.add_argument("--kld-epsilon", type=float, default=0.2, help="c3: setEpsilon (the reference uses 0.2: a few hundred particles)")
    ap.add_argument("--kld-bin", type=float, default=0.1, help="c3: setBinSize (m and rad; the reference uses 0.1)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-flush", action="store_true", help="debug only: do not flush L2 between steps")
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"],
                    help="N>1: how the crop box and the raw weights travel between the GPUs: 'peer' = stores over NVLink from the "
                         "producing kernels into CUDA-IPC windows (no collective call per frame), 'nccl' = ncclAllReduce/ncclAllGather")
    ap.add_argument("--devices", default=None, help="single-process multi-device mode (not the driver's launch): ONE process, ONE tracker object "
                                                   "per tracked object, driving these GPUs (e.g. 0,1; first = this process's device) through "
                                                   "pft_tracker_set_devices; the workload is sharded as with --gpus N under torchrun")
    ap.add_argument("--scene", default=None, choices=["peer", "replicate", "broadcast"],
                    help="N>1: how the downsampled scene reaches every GPU: 'peer' = rank 0 owns the sensor (one upload + downsample per "
                         "frame for the whole job) and its push kernel stores the result into every rank's cloud over NVLink (default "
                         "with --exchange peer); 'broadcast' = the same with ncclBroadcast (default with --exchange nccl); 'replicate' = "
                         "every rank uploads and downsamples the frame itself")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")
        return reference_arm(args)
    if args.workload == "c1":
        print("bench.py: c1 is the CPU configuration (BASELINE configs[0]): use --impl reference --workload c1", file=sys.stderr)
        return 2

    import torch
    import torch.distributed as dist
    from pcl_tracking_b200 import build as pft_build
    rank, world, local_rank = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            print("bench.py: --gpus %d needs torchrun (WORLD_SIZE=%d)" % (args.gpus, world), file=sys.stderr)
            return 2
    if not torch.cuda.is_available():
        print("bench.py: no CUDA device; the tracker has no CPU fallback (use --impl reference for the CPU arm)", file=sys.stderr)
        return 3
    if rank == 0:
        pft_build.build()
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist.barrier()
    from pcl_tracking_b200 import pcl

    ctx = pcl.Context(local_rank)
    scene_mode = args.scene or ("peer" if args.exchange == "peer" else "broadcast")
    use_nccl = world > 1 and (args.exchange == "nccl" or scene_mode == "broadcast")
    uid = None
    if use_nccl:
        box = [pcl.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        uid = box[0]
        ctx.commInit(world, rank, uid)
    stream = torch.cuda.ExternalStream(ctx.stream, device=torch.device("cuda", local_rank))
    rig = Rig(args, torch, dist, ctx, stream, rank, world, local_rank, uid)
    if args.workload in ("c5", "qhd") and world > 1:
        print("bench.py: the %s workload runs on one GPU" % args.workload, file=sys.stderr)
        return 2

    head = run_workload(rig, args.workload, args.steps, args.warmup, dump_dir=args.dump_outputs)
    line = None
    if rank == 0:
        line = {"metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": world * (len(args.devices.split(",")) if args.devices else 1), "steps": args.steps, "warmup": head["warmup"],
                "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": head["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic"}
        line.update({k: v for k, v in head.items() if k not in line})
    # ---- the other BASELINE configs, in the same line (each with its own value / e2e / roofline / clocks)
    also = args.also
    if also is None:
        also = "c4,c3,c5,qhd" if world == 1 else "c4"
    extra = [w for w in also.split(",") if w and w != "none" and w != args.workload]
    if args.workload != "c2":
        extra = []
    others = {}
    for w in extra:
        if world > 1 and w in ("c5", "qhd"):
            continue
        sub_steps = max(3, min(args.steps, 60 if w != "c4" else 30))
        try:
            r = run_workload(rig, w, sub_steps, min(args.warmup, 5), with_pipelined=False)
        except Exception as e:  # the headline stands on its own
            r = {"failed": repr(e)}
        if rank == 0:
            others[w] = r
    if rank == 0 and others:
        line["workloads"] = others
    if world > 1:
        dist.barrier()
    # ---- CPU baseline beside it (rank 0, N=1 only): bounded sample on the box's host cores
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        frames, oid0 = rig.frames(1, "sd")
        try:
            r = run_cpu(frames, oid0, PARTICLES_PER_GPU, steps=8, warmup=1, budget_s=20.0)
            line["cpu_baseline"] = {"value": r["evals_per_s"], "unit": UNIT, "cores": r["cores"], "kind": "port", "sample": r["sample"],
                                    "frames_per_s": r["frames_per_s"], "stage_s": r["stage_s"]}
        except Exception as e:  # the GPU number stands on its own
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": "failed: %r" % (e,)}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
