#!/usr/bin/env python
"""Benchmark of the per-frame hot path (YOLOv8n detect -> DeepSORT track) on B200.

    python bench.py --gpus N --steps K --warmup W            # this build, one rank per GPU
    python bench.py --impl reference --steps K --warmup W    # CPU restatement of the reference path
    python bench.py --config clip|sweep|crowded ...          # the other BASELINE.json configs (N = 1)

--config streams64 (default; BASELINE.json configs[1], and configs[2] at N = 8): a step is one pass of the hot path
over one batch: one 1080p frame of each of the 64 streams a GPU owns, no collective on the data path (weak scaling).
One JSON line is printed by rank 0.
  value     tracked frames/s, whole job, frames already resident in HBM (packed BGR, the reference's frame format),
            device-timed (CUDA events), max over ranks
  e2e       same metric through the public API with HOST frames: every step copies its frames from pinned host
            memory and reads the track table back.  The host frames are NV12 surfaces (what a hardware video
            decoder hands over, 1.5 B/pixel; aicam_preprocess_nv12 / aicam_reid_crops_nv12 produce bit for bit what
            the BGR entry points produce from the cv2-converted frame); e2e_bgr is the same with packed BGR frames
  roofline  the tcgen05 convolution kernels: algorithmic FLOPs / event-timed kernel time vs the measured bf16 peak
  cpu_baseline  the CPU restatement of the reference path (oracle nets + the reference's own tracker when
            oracle/_ref is built) on the box's host cores
--config clip (configs[0]): the reference's own 960x540 clip, one stream, batch 1, through the reference-shaped
facades (YOLODetector.detect -> DeepSORT.update), timed the reference's way (frames / sum of detect + update wall time,
/root/reference/src/aicamera_tracker.py:175,199-207) plus p50 / p99 per-frame latency.
--config sweep (configs[3]): YOLOv8 n / s / m detection-only (K1-K4), batch 1-256, against the tensor-pipe roofline.
--config crowded (configs[4]): 300 persons per frame per stream: ReID batch 300 per stream and a 300 x 300
association per stream through TrackingPipeline (planted person boxes riding on the moving texture; the detector still
runs and is timed).

--dump-outputs DIR (--config streams64): after the timed steps, rank 0 writes what TrackingPipeline.step returned in the
last timed step as DIR/out_tracks.npy (float64 [S, T, 6]: x1, y1, x2, y2, id, class), DIR/out_conf.npy (float32 [S, T])
and DIR/out_count.npy (float64 [S]).  Rows at or past a stream's count hold no track and are written as zeros.  The
inputs depend only on the arguments, so two builds run with the same arguments can be compared file for file.

--steps sets the number of timed steps of --config streams64 and crowded and of --impl reference.  --config clip
times the whole clip (and 128 device-resident steps), --config sweep fixed iteration counts per batch size.

The benchmark writes nothing into the repository, so it also runs from a read-only checkout: the seeded weight blobs go
to $AICAM_BLOB_DIR when it is set, else to a temporary directory removed at exit (regenerating them takes a few
seconds, outside every timed region).
"""
import argparse
import atexit
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import threading
import time

sys.dont_write_bytecode = True  # nothing into the tree, not even __pycache__ for the modules build() never imported
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

STREAMS_PER_GPU = 64
FRAME_HW = (1080, 1920)
TARGET_DETS = 16.0
RING = 12
METRIC = "tracked_frames_per_sec"
WORKLOAD = "YOLOv8n+DeepSORT-ReID, 64 synthetic 1080p streams per GPU, ~16 tracked detections/frame"
CLIP_PATH = os.path.join(ROOT, "tests", "golden", "aicamera_test_clip.mp4")
CLIP_WORKLOAD = "YOLOv8n+DeepSORT-ReID on assets/aicamera_test_clip.mp4 (960x540, 500 frames), single stream, batch 1"
TRAFFIC_JSON = os.path.join(ROOT, "profiles", "r2_step_traffic.json")


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return dict(hbm=p["hbm_gbs"], bf16=p.get("bf16_tflops_sustained", p["bf16_tflops"]), bf16_burst=p["bf16_tflops"],
                    source="measured")
    except Exception:
        return dict(hbm=6650.0, bf16=1400.0, bf16_burst=1590.0, source="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for n, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------------------------------------
# CPU legs (the only places that execute oracle/)
# ---------------------------------------------------------------------------------------------------------------------
def make_cpu_pipeline(yolo_blob, reid_blob, bias):
    """One stream of the reference path on the CPU: oracle nets (the reference's TensorRT engines and ONNX files do
    not exist here) + the REAL reference DeepSORT when oracle/_ref is built, else its restatement."""
    from oracle import ref_bridge
    from oracle.pipeline import Pipeline, ReID
    p = Pipeline(yolo_blob, reid_blob, yolo_bias=bias)
    kind = "port"
    if ref_bridge.available():
        p.tracker = ref_bridge.RefDeepSORT(ReID(reid_blob))
        kind = "reference"
    return p, kind


def cpu_baseline_run(yolo_blob, reid_blob, bias, frames_by_stream, steps, warmup=0):
    """CPU pipeline (one instance per stream, as one reference process per stream) over `steps` time steps of the
    given host frames.  Returns (frames/s, seconds, cores, tracker kind)."""
    import torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    made = [make_cpu_pipeline(yolo_blob, reid_blob, bias) for _ in frames_by_stream]
    pipes, kind = [m[0] for m in made], made[0][1]
    n = 0
    t0 = None
    for t in range(warmup + steps):
        if t == warmup:
            t0 = time.perf_counter()
        for s, fr in enumerate(frames_by_stream):
            pipes[s].step(fr[t % len(fr)])
            n += t >= warmup
    dt = time.perf_counter() - t0
    return n / dt, dt, cores, kind


def clip_frames(n=0):
    from ai_camera_b200.aicamera_tracker import video_frames
    if not os.path.exists(CLIP_PATH):
        raise RuntimeError("clip fixture missing: python tests/golden/make_clip_fixture.py")
    return list(video_frames(CLIP_PATH, n))


def run_reference(args):
    """--impl reference: the CPU restatement of the reference path (the reference's own runtime, TensorRT + its ONNX
    files, is not available; SURVEY.md 0.1-0.2) with the reference's real tracker (oracle/_ref) underneath."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch  # noqa: F401
    from ai_camera_b200 import synth
    yolo, reid = synth.make_blobs(synth.blob_dir())
    if args.config == "clip":
        bias = synth.shifted_class_bias(yolo, synth.CLIP_LOGIT_SHIFT)
        frames = [clip_frames(args.warmup + args.steps)]
        workload, sample = CLIP_WORKLOAD, "the first %d clip frames" % (args.warmup + args.steps)
        n_sample = 1
    elif args.config in ("sweep", "crowded"):
        emit({"impl": "reference", "unavailable": "--config %s has no separate reference arm; see its cpu_baseline" % args.config})
        return
    else:
        bias = synth.shifted_class_bias(yolo)
        n_sample = 2  # streams sampled per step (a bounded sample of the 64-stream batch)
        video = synth.SynthVideo(n_sample, FRAME_HW, n_frames=6, device="cpu")
        frames = [[video.ring[t, s].numpy() for t in range(video.n_frames)] for s in range(n_sample)]
        workload, sample = WORKLOAD, "%d of %d streams per step" % (n_sample, STREAMS_PER_GPU)
    fps, dt, cores, kind = cpu_baseline_run(yolo, reid, bias, frames, args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / max(1, args.steps),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload, "sample": sample,
                   "runtime": "PyTorch-CPU fp32 restatement of the two nets (oracle port) + %s" % (
                       "the reference's own DeepSORT / TrackerCore (oracle/_ref)" if kind == "reference" else "numpy/scipy tracker port")},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port", "tracker_kind": kind,
                         "sample": "%d stream(s) x %d steps (%s)" % (n_sample, args.steps, sample)},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


_RESULT = None  # the real stdout; everything else written to file descriptor 1 (NCCL's version banner, library chatter) goes to stderr


def emit(line):
    _RESULT.write(json.dumps(line) + "\n")
    _RESULT.flush()


def pin_rank(local, world):
    """Give every rank its own contiguous share of the cores this process may run on (launch thread and copy
    engine callbacks stay put; the pinned host ring is then first-touched from those cores)."""
    try:
        cpus = sorted(os.sched_getaffinity(0))
        share = len(cpus) // max(1, world)
        if world > 1 and share >= 2:
            os.sched_setaffinity(0, cpus[local * share:(local + 1) * share])
    except Exception:
        pass


def dump_outputs(directory, out_tracks, out_conf, out_count):
    """Host copies of one step's track tables -> DIR/<name>.npy; rows past each stream's count are zeroed (they are
    left over from earlier steps, not part of the result)."""
    import numpy as np
    tracks, conf, count = (t.cpu().numpy() for t in (out_tracks, out_conf, out_count))
    valid = np.arange(tracks.shape[1])[None, :] < count[:, None]
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "out_tracks.npy"), np.where(valid[..., None], tracks, 0).astype(np.float64))
    np.save(os.path.join(directory, "out_conf.npy"), np.where(valid, conf, 0).astype(np.float32))
    np.save(os.path.join(directory, "out_count.npy"), count.astype(np.float64))


def conv_roofline(lib, _lib, one_step, crops_of_step, flops_of, prof_steps=6):
    """Event-instrumented pass over the tcgen05 convolution kernels: (TFLOP/s, ms per step, launches per step, crops)."""
    lib.aicam_profile_enable(1)
    crops = 0.0
    for _ in range(prof_steps):
        one_step()
        crops += crops_of_step()
    crops /= prof_steps
    ms, nl = _lib.C.c_double(), _lib.C.c_uint64()
    _lib.check(lib.aicam_profile_conv(_lib.C.byref(ms), _lib.C.byref(nl)))
    lib.aicam_profile_enable(0)
    conv_ms = ms.value / prof_steps
    flops = flops_of(crops)
    return (flops / (conv_ms * 1e-3) / 1e12 if conv_ms > 0 else 0.0), conv_ms, max(1, nl.value // prof_steps), crops, flops


def roofline_entry(kernel, achieved, conv_ms, launches, crops, flops, prof_steps):
    peaks = measured_peaks()
    traffic = None
    try:
        with open(TRAFFIC_JSON) as f:
            traffic = json.load(f)
    except Exception:
        pass
    return {"kernel": kernel, "bound": "tensor", "achieved": achieved, "peak": peaks["bf16"], "unit": "TFLOP/s",
            "frac": achieved / peaks["bf16"],
            "traffic": (traffic["dram_bytes"] / traffic["launches"]) if traffic else None, "traffic_unit": "bytes/launch",
            "traffic_detail": traffic, "peak_source": peaks["source"] + " (bf16_tflops_sustained: the kernels run inside a ms-long step)",
            "launches_per_step": int(launches), "avg_launch_us": 1e3 * conv_ms / launches, "flops_per_launch": flops / launches,
            "kernel_ms_per_step": conv_ms, "flops_per_step": flops, "crops_per_profiled_step": crops, "profiled_steps": prof_steps}


# ---------------------------------------------------------------------------------------------------------------------
# configs[1] / configs[2]: 64 streams per GPU
# ---------------------------------------------------------------------------------------------------------------------
def run_streams(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    pin_rank(local, world)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)

    from ai_camera_b200 import _lib, sharding, synth
    from ai_camera_b200.pipeline import TrackingPipeline
    lib = _lib.load()
    S = args.streams
    H, W = FRAME_HW
    blob_dir = synth.blob_dir()
    if rank == 0:
        synth.make_blobs(blob_dir)
    if world > 1:
        dist.barrier()
    yolo, reid = synth.make_blobs(blob_dir)
    first_stream, _ = sharding.stream_partition(S * world, world, rank)  # weak scaling: S streams per GPU
    video = synth.SynthVideo(S, FRAME_HW, n_frames=RING, device=dev, first_stream=first_stream)
    # The same video as NV12 surfaces (the e2e leg's host format).  The BGR ring is then RE-DERIVED from the NV12 ring
    # with the path's own converter (== cv2 COLOR_YUV2BGR_NV12), so both formats hold exactly the same pixels and
    # the two legs do identical work downstream of K1 / K5.
    nv12_ring = torch.empty((RING, S, H * 3 // 2, W), dtype=torch.uint8, device=dev)
    for k in range(RING):
        nv12_ring[k] = synth.bgr_to_nv12(video.ring[k])
        _lib.check(lib.aicam_nv12_to_bgr(_lib.ptr(nv12_ring[k]), S, H, W, _lib.ptr(video.ring[k]), _lib.stream_ptr(dev)))
    torch.cuda.synchronize(dev)
    pipe = TrackingPipeline(yolo, reid, S, dev, max_tracks=128, max_crops=S * 40)
    delta = synth.DEFAULT_LOGIT_SHIFT
    bias = synth.shifted_class_bias(yolo, delta)
    synth.apply_class_bias(pipe.detector.engine, bias)

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    # ---- device-resident run ----------------------------------------------------------------
    step_no = [0]

    def one_step():
        out = pipe.step(video.frames(step_no[0]))
        step_no[0] += 1
        return out

    pipe.tracker.count_stats = True  # device-side totals of crops / reported tracks (two tiny torch adds per step)
    for _ in range(args.warmup):
        one_step()
    counted0 = lib.aicam_launch_count()
    one_step()
    launches_counted = lib.aicam_launch_count() - counted0  # kernels of ONE step, counted by the library itself
    torch.cuda.synchronize(dev)
    # CUDA graphs: one graph per ring position (the frame pointer is baked into the graph)
    graphs = None
    if not args.no_graph:
        try:
            graphs = []
            stream = torch.cuda.Stream(dev)
            with torch.cuda.stream(stream):
                for k in range(RING):
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g, stream=stream):
                        pipe.step(video.ring[k])
                    graphs.append(g)
            torch.cuda.synchronize(dev)
        except Exception as e:  # capture unsupported -> eager launches
            sys.stderr.write("cuda graph capture failed (%s); running eager\n" % e)
            graphs = None
            torch.cuda.synchronize(dev)

    def timed_step():
        if graphs is None:
            return one_step()
        graphs[video.index(step_no[0])].replay()
        step_no[0] += 1

    for _ in range(3):
        timed_step()
    sync_all()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = lib.aicam_launch_count()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    pipe.tracker.crop_total.zero_()
    pipe.tracker.track_total.zero_()
    sync_all()
    ev[0].record()
    for k in range(args.steps):
        timed_step()
        ev[k + 1].record()
    torch.cuda.synchronize(dev)
    total_ms = ev[0].elapsed_time(ev[-1])
    per_step = [ev[k].elapsed_time(ev[k + 1]) for k in range(args.steps)]
    if args.dump_outputs and rank == 0:  # the buffers TrackingPipeline.step returns (and the graphs write into)
        dump_outputs(args.dump_outputs, pipe.tracker.out_tracks, pipe.tracker.out_conf, pipe.tracker.out_count)
    sync_all()
    launches_eager = launches_counted
    gpu_launches = (lib.aicam_launch_count() - launches0) if graphs is None else launches_eager * args.steps
    crops_per_step = float(pipe.tracker.crop_total.item()) / args.steps      # mean over the timed steps
    tracks_out = float(pipe.tracker.track_total.item()) / args.steps
    overflow = int(pipe.tracker.overflow().any())

    # ---- end to end: host frames in, track tables out, every step -------------------------
    T = pipe.tracker.T
    host_out = [torch.empty((S, T, 6), dtype=torch.int32).pin_memory(),
                torch.empty((S, T), dtype=torch.float32).pin_memory(), torch.empty(S, dtype=torch.int32).pin_memory()]
    copy_stream = torch.cuda.Stream(dev)
    e2e_steps = max(4, min(args.steps, 20))

    def e2e_measure(ring):
        host_ring = [ring[k].cpu().pin_memory() for k in range(min(4, RING))]
        dev_in = [torch.empty_like(ring[0]) for _ in range(2)]

        def e2e_run(n):
            # double buffering: the H2D copy of step k+1 overlaps the compute of step k
            ready = [torch.cuda.Event(), torch.cuda.Event()]
            done = [torch.cuda.Event(), torch.cuda.Event()]
            with torch.cuda.stream(copy_stream):
                dev_in[0].copy_(host_ring[0], non_blocking=True)
                ready[0].record()
            for k in range(n):
                cur, nxt = k & 1, (k + 1) & 1
                if k + 1 < n:
                    with torch.cuda.stream(copy_stream):
                        if k >= 1:
                            copy_stream.wait_event(done[nxt])
                        dev_in[nxt].copy_(host_ring[(k + 1) % len(host_ring)], non_blocking=True)
                        ready[nxt].record()
                torch.cuda.current_stream(dev).wait_event(ready[cur])
                ot, oc, on = pipe.step(dev_in[cur])
                host_out[0].copy_(ot, non_blocking=True)
                host_out[1].copy_(oc, non_blocking=True)
                host_out[2].copy_(on, non_blocking=True)
                done[cur].record()
            torch.cuda.synchronize(dev)

        e2e_run(3)
        sync_all()
        # timed on the device: the start event precedes the first copy's stream (the copy stream waits on it), the
        # end event follows the last device-to-host copy on the compute stream
        ee0, ee1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ee0.record()
        copy_stream.wait_event(ee0)
        e2e_run(e2e_steps)
        ee1.record()
        torch.cuda.synchronize(dev)
        secs = ee0.elapsed_time(ee1) * 1e-3
        sync_all()
        del host_ring, dev_in
        return secs, ring[0].numel()

    e2e_s, h2d = e2e_measure(nv12_ring)
    e2e_bgr_s, h2d_bgr = e2e_measure(video.ring)
    clocks = sampler.stop() if rank == 0 else None
    d2h = sum(t.numel() * t.element_size() for t in host_out)

    # ---- roofline of the convolution kernels (separate, event-instrumented pass) -------------
    prof_steps = 6
    achieved, conv_ms, launches_step, prof_crops, flops_step = conv_roofline(
        lib, _lib, one_step, lambda: float(pipe.tracker.crop_count[0].item()),
        lambda crops: S * pipe.detector.engine.flops_per_item() + crops * pipe.tracker.reid.flops_per_item(), prof_steps)

    # ---- gather (the only collective: final stats) -------------------------------------------
    allst = np.asarray(sharding.gather_stats([total_ms, e2e_s, crops_per_step, float(tracks_out), float(overflow), e2e_bgr_s], dev))
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    max_ms = float(allst[:, 0].max())
    max_e2e = float(allst[:, 1].max())
    max_e2e_bgr = float(allst[:, 5].max())
    frames_total = world * S * args.steps
    value = frames_total / (max_ms * 1e-3)
    line = {
        "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": max_ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": WORKLOAD, "streams_per_gpu": S, "frame": "1080x1920x3 u8",
                   "crops_per_step": float(allst[:, 2].mean()), "tracks_reported_per_step": float(allst[:, 3].mean()),
                   "detections_per_frame": float(allst[:, 2].mean()) / S,
                   "tracker_overflow": bool(allst[:, 4].any()), "l2": "inputs larger than L2 (398 MB of frames per step)",
                   "cuda_graph": graphs is not None, "detector_logit_shift": delta,
                   "weights": "seeded synthetic (no checkpoints offline)",
                   "e2e_input": "NV12 host surfaces (decoder output format, 199 MB per step); e2e_bgr: packed BGR host frames (398 MB per step)"},
        "p50_latency_ms": statistics.median(per_step),
        "step_ms_distribution": {"min": min(per_step), "p10": sorted(per_step)[len(per_step) // 10], "p50": statistics.median(per_step),
                                 "p90": sorted(per_step)[(9 * len(per_step)) // 10], "max": max(per_step),
                                 "first_8": [round(x, 3) for x in per_step[:8]],
                                 **({"all": [round(x, 2) for x in per_step]} if os.environ.get("AICAM_BENCH_DUMP_STEPS") else {}),
                                 "note": "rank 0, per-step CUDA events inside the timed region; value uses the whole region (mean)"},
        "clocks": clocks,
        "e2e": {"value": world * S * e2e_steps / max_e2e, "unit": "frames/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "steps": e2e_steps, "h2d_gbs": h2d * e2e_steps / max_e2e / 1e9, "input": "nv12",
                "note": "NV12 frames from pinned host memory through TrackingPipeline.step, copy double-buffered against "
                        "compute; track tables copied back every step"},
        "e2e_bgr": {"value": world * S * e2e_steps / max_e2e_bgr, "unit": "frames/s", "h2d_bytes_per_step": h2d_bgr,
                    "d2h_bytes_per_step": d2h, "steps": e2e_steps, "h2d_gbs": h2d_bgr * e2e_steps / max_e2e_bgr / 1e9,
                    "note": "packed BGR host frames (the reference's frame format): bounded by the PCIe host-to-device rate"},
        "gpu_launches": int(gpu_launches),
        "roofline": roofline_entry("tcgen05 convolution kernels: conv_win_kernel + conv_pair_kernel + reid_stem_pool_kernel "
                                   "(all %d launches of a step)" % launches_step, achieved, conv_ms, launches_step, prof_crops,
                                   flops_step, prof_steps),
    }
    if world == 1 and not args.no_cpu_baseline:
        n_sample, cpu_steps = 8, 16  # ~10 s of host work: a bounded sample of the 64-stream workload
        frames = [[video.ring[t, s].cpu().numpy() for t in range(min(RING, 8))] for s in range(n_sample)]
        fps, dt, cores, kind = cpu_baseline_run(yolo, reid, bias, frames, cpu_steps, warmup=1)
        line["cpu_baseline"] = {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port", "tracker_kind": kind,
                                "sample": "%d streams x %d steps of the same 1080p frames (%.1f s)" % (n_sample, cpu_steps, dt)}
    emit(line)
    if world > 1:
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------------------------
# configs[0]: the reference's clip, single stream, batch 1
# ---------------------------------------------------------------------------------------------------------------------
def run_clip(args):
    import numpy as np
    import torch
    from ai_camera_b200 import _lib, synth
    from ai_camera_b200.aicamera_tracker import run_single_stream
    from ai_camera_b200.deepsort_tracker import DeepSORT
    from ai_camera_b200.pipeline import TrackingPipeline
    from ai_camera_b200.yolo_detector import YOLODetector
    lib = _lib.load()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    yolo, reid = synth.make_blobs(synth.blob_dir())
    bias = synth.shifted_class_bias(yolo, synth.CLIP_LOGIT_SHIFT)
    frames = clip_frames()
    H, W = frames[0].shape[:2]
    det = YOLODetector(yolo)
    synth.apply_class_bias(det.trt_engine, bias)
    trk = DeepSORT(reid)
    n_tracks = [0]

    def on_frame(i, f, d, tr):
        n_tracks[0] += len(tr)
    # warm-up (tracks stay: the loop continues).  The first frame runs eagerly through the library, which counts its launches; from
    # the third call on the facades replay a CUDA graph of the same launches (the library's counter does not see replays)
    l0 = lib.aicam_launch_count()
    run_single_stream(frames[:1], det, trk, on_frame)
    launches_per_frame = lib.aicam_launch_count() - l0
    run_single_stream(frames[1:max(3, args.warmup)], det, trk, on_frame)
    n_tracks[0] = 0
    sampler = ClockSampler(0)
    sampler.start()
    launches0 = lib.aicam_launch_count()
    stats = run_single_stream(frames, det, trk, on_frame)
    launches = max(lib.aicam_launch_count() - launches0, launches_per_frame * stats.frames)
    clocks = sampler.stop()
    s = stats.summary()
    # device-resident single-stream number: the same frames through a 1-stream TrackingPipeline, no host round trip
    pipe = TrackingPipeline(yolo, reid, 1, dev, max_tracks=256, max_crops=128)
    synth.apply_class_bias(pipe.detector.engine, bias)
    dframes = torch.from_numpy(np.stack(frames[:128])).to(dev)
    for k in range(8):
        pipe.step(dframes[k:k + 1])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(128):
        pipe.step(dframes[k:k + 1])
    e1.record()
    torch.cuda.synchronize()
    dev_ms = e0.elapsed_time(e1) / 128
    k = [0]

    def one_step():
        pipe.step(dframes[k[0] % 128:k[0] % 128 + 1])
        k[0] += 1
    achieved, conv_ms, launches_step, prof_crops, flops_step = conv_roofline(
        lib, _lib, one_step, lambda: float(pipe.tracker.crop_count[0].item()),
        lambda crops: pipe.detector.engine.flops_per_item() + crops * pipe.tracker.reid.flops_per_item(), 6)
    line = {
        "metric": METRIC, "value": 1e3 / dev_ms, "unit": "frames/s", "n_gpus": 1, "steps": len(frames), "warmup": max(3, args.warmup),
        "ms_per_step": dev_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "the reference's clip (tests/golden/aicamera_test_clip.mp4), seeded synthetic weights",
        "config": {"workload": CLIP_WORKLOAD, "frame": "%dx%dx3 u8" % (H, W), "detector_logit_shift": synth.CLIP_LOGIT_SHIFT,
                   "tracks_reported_per_frame": n_tracks[0] / max(1, stats.frames),
                   "value_is": "1-stream TrackingPipeline on device-resident frames, CUDA events; e2e is the facade loop"},
        "p50_latency_ms": s["p50_ms"], "p99_latency_ms": s["p99_ms"], "clocks": clocks,
        "e2e": {"value": s["avg_fps"], "unit": "frames/s", "h2d_bytes_per_step": H * W * 3, "d2h_bytes_per_step": 4 * (1 + 6 * 100) + 4 * (1 + 7 * 256),
                "steps": stats.frames, "p50_ms": s["p50_ms"], "p99_ms": s["p99_ms"],
                "note": "YOLODetector.detect(numpy frame) -> DeepSORT.update(...) per frame, wall clock of detect + update as the "
                        "reference accounts it (aicamera_tracker.py:175,199-207); one frame upload, two host synchronisations per frame"},
        "gpu_launches": int(launches),
        "roofline": roofline_entry("tcgen05 convolution kernels at batch 1 (latency-bound by construction)", achieved, conv_ms,
                                   launches_step, prof_crops, flops_step, 6),
    }
    if not args.no_cpu_baseline:
        n = 60
        fps, dt, cores, kind = cpu_baseline_run(yolo, reid, bias, [frames[:n + 2]], n, warmup=2)
        line["cpu_baseline"] = {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port", "tracker_kind": kind,
                                "sample": "the first %d clip frames (%.1f s)" % (n, dt)}
    emit(line)


# ---------------------------------------------------------------------------------------------------------------------
# configs[3]: YOLOv8 n / s / m detection-only sweep
# ---------------------------------------------------------------------------------------------------------------------
def run_sweep(args):
    import torch
    from ai_camera_b200 import _lib, synth, weights as Wt
    from ai_camera_b200.pipeline import BatchDetector
    lib = _lib.load()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    peaks = measured_peaks()
    rows = []
    best = None
    sampler = ClockSampler(0)
    sampler.start()
    launches0 = lib.aicam_launch_count()
    for sc in args.scales:
        path = os.path.join(synth.blob_dir(), "yolov8%s_sweep.aicw" % sc)
        if not os.path.exists(path):
            os.makedirs(os.path.dirname(path), exist_ok=True)
            Wt.write_blob(path, *Wt.synth_yolov8_weights(sc, seed=0))
        det = BatchDetector(path, args.max_batch, dev)
        flops = det.engine.flops_per_item()
        b = 1
        while b <= args.max_batch:
            x = torch.randint(0, 256, (b, 640, 640, 3), dtype=torch.uint8, device=dev)
            for _ in range(3):
                det.detect(x)
            iters = 10 if b <= 32 else 4
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(iters):
                det.detect(x)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / iters
            lib.aicam_profile_enable(1)
            det.detect(x)
            cm, nl = _lib.C.c_double(), _lib.C.c_uint64()
            _lib.check(lib.aicam_profile_conv(_lib.C.byref(cm), _lib.C.byref(nl)))
            lib.aicam_profile_enable(0)
            tf = flops * b / (cm.value * 1e-3) / 1e12 if cm.value > 0 else 0.0
            row = {"model": "yolov8" + sc, "batch": b, "ms": ms, "frames_per_s": b / ms * 1e3, "conv_kernel_ms": cm.value,
                   "conv_tflops": tf, "frac_of_bf16_peak": tf / peaks["bf16"]}
            rows.append(row)
            sys.stderr.write("%(model)s b=%(batch)d %(ms).3f ms %(frames_per_s).0f fps conv %(conv_tflops).1f TFLOP/s\n" % row)
            if best is None or row["conv_tflops"] > best["conv_tflops"]:
                best = row
            del x
            b *= 2
        del det
        torch.cuda.empty_cache()
    clocks = sampler.stop()
    head = max((r for r in rows if r["model"] == "yolov8" + args.scales[-1]), key=lambda r: r["frames_per_s"])
    line = {
        "metric": "detection_frames_per_sec", "value": head["frames_per_s"], "unit": "frames/s", "n_gpus": 1, "steps": len(rows), "warmup": 3,
        "ms_per_step": head["ms"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": "YOLOv8 %s 640x640 detection-only (K1-K4: preprocess, network, decode, NMS), batch 1-%d; value = %s at batch %d" % (
            "/".join(args.scales), args.max_batch, head["model"], head["batch"]), "weights": "seeded synthetic"},
        "clocks": clocks, "sweep": rows,
        "e2e": {"value": head["frames_per_s"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                "note": "device-resident input; the sweep isolates the detector (see --config streams64 for host-fed numbers)"},
        "gpu_launches": int(lib.aicam_launch_count() - launches0),
        "roofline": {"kernel": "tcgen05 convolution kernels of %s at batch %d" % (best["model"], best["batch"]), "bound": "tensor",
                     "achieved": best["conv_tflops"], "peak": peaks["bf16"], "unit": "TFLOP/s", "frac": best["frac_of_bf16_peak"],
                     "traffic": None, "peak_source": peaks["source"]},
    }
    emit(line)


# ---------------------------------------------------------------------------------------------------------------------
# configs[4]: crowded scene, 300 persons per frame per stream
# ---------------------------------------------------------------------------------------------------------------------
def run_crowded(args):
    import numpy as np
    import torch
    from ai_camera_b200 import _lib, synth
    from ai_camera_b200.pipeline import TrackingPipeline
    lib = _lib.load()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    S, D = args.streams if args.streams != STREAMS_PER_GPU else 16, args.persons
    H, W = FRAME_HW
    yolo, reid = synth.make_blobs(synth.blob_dir())
    ring = 8
    video = synth.SynthVideo(S, FRAME_HW, n_frames=ring, device=dev)
    pipe = TrackingPipeline(yolo, reid, S, dev, max_tracks=D + 84, max_crops=S * D, topk=D)
    synth.apply_class_bias(pipe.detector.engine, synth.shifted_class_bias(yolo))
    trk = pipe.tracker
    # planted persons: a grid of boxes that ride on the stream's moving texture (so that every person keeps its
    # appearance and its constant velocity), jittered by a pixel; the detector runs on the frame as usual (timed) but
    # the tracker is fed the planted boxes (SURVEY.md 8d: random-init heads give no usable persons)
    g = torch.Generator(device="cpu").manual_seed(7)
    cols = int(np.ceil(np.sqrt(D * W / H)))
    rows_ = int(np.ceil(D / cols))
    cw, ch = (W - 160) / cols, (H - 160) / rows_
    idx = torch.arange(D)
    cx0 = (80 + (idx % cols + 0.5) * cw).to(dev)
    cy0 = (80 + (idx // cols + 0.5) * ch).to(dev)
    bw, bh = min(0.8 * cw, 48.0), min(0.9 * ch, 96.0)
    vel = torch.tensor(video.velocity, dtype=torch.float32, device=dev) * 3.0  # source pixels per ring index
    scores = torch.full((S, D), 0.9, dtype=torch.float32, device=dev)
    labels = torch.zeros((S, D), dtype=torch.int32, device=dev)
    num = torch.full((S,), D, dtype=torch.int32, device=dev)
    boxes = torch.zeros((S, D, 4), dtype=torch.float32, device=dev)
    jit = torch.randn((64, S, D, 4), generator=g).to(dev)
    step_no = [0]

    def one_step():
        k = video.index(step_no[0])
        # the texture moves by -velocity * index (frame k shows tex[oy + 3 vy k ...]): objects move the opposite way
        x = cx0[None, :] - vel[:, 0:1] * k
        y = cy0[None, :] - vel[:, 1:2] * k
        boxes.copy_(torch.stack([x - bw / 2, y - bh / 2, x + bw / 2, y + bh / 2], dim=-1) + jit[step_no[0] % 64])
        frames = video.ring[k]
        pipe.detector.detect(frames)
        out = trk.update(frames, num, boxes, scores, labels)
        step_no[0] += 1
        return out

    warm = max(args.warmup, 110)  # galleries fill to the budget (100) before the timed region
    for _ in range(warm):
        one_step()
    torch.cuda.synchronize()
    sampler = ClockSampler(0)
    sampler.start()
    launches0 = lib.aicam_launch_count()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    ev[0].record()
    for k in range(args.steps):
        one_step()
        ev[k + 1].record()
    torch.cuda.synchronize()
    launches = lib.aicam_launch_count() - launches0
    clocks = sampler.stop()
    total_ms = ev[0].elapsed_time(ev[-1])
    per_step = [ev[k].elapsed_time(ev[k + 1]) for k in range(args.steps)]
    reported = float(trk.out_count.float().mean().item())
    ints, _ = trk.snapshot(0)
    gal = float(ints[:, 6].mean()) if len(ints) else 0.0
    overflow = trk.overflow()
    # tracker kernels alone (filter excluded): event-timed around aicam_tracker_step with this step's inputs
    st = _lib.stream_ptr(dev)
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reid0, reid1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fwd = lib.aicam_reid_forward_nhwc8 if trk._nhwc8 else lib.aicam_reid_forward
    reid0.record()
    _lib.check(fwd(trk.reid.handle, _lib.ptr(trk.crops), trk.max_crops, _lib.ptr(trk.crop_count), _lib.ptr(trk.feats), st))
    reid1.record()
    probe = [torch.zeros((S, trk.T, D), dtype=torch.float32, device=dev) for _ in range(2)]
    ids, nt = torch.zeros((S, trk.T), dtype=torch.int32, device=dev), torch.zeros(S, dtype=torch.int32, device=dev)
    t0.record()
    _lib.check(lib.aicam_tracker_cost_probe(trk._h, _lib.ptr(boxes), D, _lib.ptr(trk.det_index), _lib.ptr(trk.det_count),
                                            _lib.ptr(trk.crop_slot), _lib.ptr(trk.feats), _lib.ptr(probe[0]), _lib.ptr(probe[1]),
                                            _lib.ptr(ids), _lib.ptr(nt), st))
    t1.record()
    torch.cuda.synchronize()
    crops = float(trk.crop_count[0].item())
    reid_ms = reid0.elapsed_time(reid1)
    reid_tf = crops * trk.reid.flops_per_item() / (reid_ms * 1e-3) / 1e12
    peaks = measured_peaks()
    frames_total = S * args.steps
    line = {
        "metric": METRIC, "value": frames_total / (total_ms * 1e-3), "unit": "frames/s", "n_gpus": 1, "steps": args.steps, "warmup": warm,
        "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic",
        "config": {"workload": "crowded scene: %d streams x %d persons per 1080p frame (ReID batch %d per stream, %d x %d association "
                               "per stream), YOLOv8n + ReID + DeepSORT through TrackingPipeline" % (S, D, D, D, D),
                   "streams": S, "persons_per_frame": D, "crops_per_step": crops, "tracks_reported_per_stream": reported,
                   "mean_gallery_size": gal, "tracker_overflow": bool(overflow.any()),
                   "detections": "planted person boxes riding on the moving texture; the detector runs and is timed, its output is not used",
                   "reid_ms_per_step": reid_ms, "appearance_probe_ms": t0.elapsed_time(t1)},
        "p50_latency_ms": statistics.median(per_step),
        "step_ms_distribution": {"min": min(per_step), "p10": sorted(per_step)[len(per_step) // 10], "p50": statistics.median(per_step),
                                 "p90": sorted(per_step)[(9 * len(per_step)) // 10], "max": max(per_step),
                                 "first_8": [round(x, 3) for x in per_step[:8]],
                                 **({"all": [round(x, 2) for x in per_step]} if os.environ.get("AICAM_BENCH_DUMP_STEPS") else {}),
                                 "note": "rank 0, per-step CUDA events inside the timed region; value uses the whole region (mean)"}, "clocks": clocks,
        "e2e": {"value": frames_total / (total_ms * 1e-3), "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                "note": "device-resident frames (the host-fed leg is measured in --config streams64)"},
        "gpu_launches": int(launches),
        "roofline": {"kernel": "ReID tcgen05 convolution kernels at %d crops" % int(crops), "bound": "tensor", "achieved": reid_tf,
                     "peak": peaks["bf16"], "unit": "TFLOP/s", "frac": reid_tf / peaks["bf16"], "traffic": None, "peak_source": peaks["source"]},
    }
    emit(line)


def positive_int(text):
    value = int(text)
    if value < 1:
        raise argparse.ArgumentTypeError("must be at least 1, got %d" % value)
    return value


def main():
    global _RESULT
    sys.stdout.flush()
    _RESULT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)  # stdout carries exactly one JSON line
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=40,
                    help="timed steps of --config streams64 / crowded and of --impl reference; --config clip times the "
                         "whole clip and --config sweep fixed iteration counts per batch size")
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--impl", default="aicam", choices=["aicam", "reference"])
    ap.add_argument("--config", default="streams64", choices=["streams64", "clip", "sweep", "crowded"])
    ap.add_argument("--streams", type=int, default=STREAMS_PER_GPU)
    ap.add_argument("--persons", type=int, default=300)
    ap.add_argument("--scales", default="nsm")
    ap.add_argument("--max-batch", type=int, default=256)
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's track tables as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "aicam" or args.config != "streams64"):
        ap.error("--dump-outputs is implemented for --impl aicam --config streams64")
    if "AICAM_BLOB_DIR" not in os.environ:
        blob_dir = tempfile.mkdtemp(prefix="aicam-bench-blobs-")
        atexit.register(shutil.rmtree, blob_dir, True)
        os.environ["AICAM_BLOB_DIR"] = blob_dir
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3)
    if args.config != "streams64" and int(os.environ.get("RANK", "0")) != 0:
        return  # the other configs are single-GPU measurements
    return {"streams64": run_streams, "clip": run_clip, "sweep": run_sweep, "crowded": run_crowded}[args.config](args)


if __name__ == "__main__":
    main()
