#!/usr/bin/env python
"""Cost and saving of per-stream regions: 64 synthetic 1080p BGR streams (synth.SynthVideo, the detector calibrated with
synth.shifted_class_bias), graphed list steps (captured once, replayed after frame_table.set):
  (a) no regions;
  (b) every stream with a pass-all region at the maxima: one full-frame include and seven exclude polygons off the frame,
      8 x 32 vertices - the most test work a step can do, with outputs identical to (a), so b - a is the region test's cost;
  (c) every stream excluding the top half of its frame: fewer crops and ReID rows per step (a different workload).
Paths are timed in alternating rounds in one process (CUDA events, median over rounds).  Then region_kernel and
filter_kernel alone: eager (b) steps under torch.profiler with CUDA activities.  One JSON line.
    python scripts/region_bench.py [--steps N] [--rounds R] [--warmup W]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ai_camera_b200 import synth  # noqa: E402
from ai_camera_b200.pipeline import StreamSettings, TrackingPipeline  # noqa: E402

LIMIT = 1 << 20


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = (x.strip() for x in q.split(","))
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # the numbers stand without it, but say so
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": "unknown (%s)" % e}


def pass_all():
    """One include of 32 vertices around the whole coordinate range, seven excludes of 32 vertices left of every frame."""
    step = 2 * LIMIT // 8
    ring = ([(-LIMIT + k * step, -LIMIT) for k in range(8)] + [(LIMIT, -LIMIT + k * step) for k in range(8)] +
            [(LIMIT - k * step, LIMIT) for k in range(8)] + [(-LIMIT, LIMIT - k * step) for k in range(8)])
    off = [[(-5000 - 10 * k - j, -100 - (j * j) % 50) for j in range(32)] for k in range(7)]
    return StreamSettings(include_regions=[ring], exclude_regions=off)


def top_half(w=1920, h=1080):
    return StreamSettings(exclude_regions=[((0, 0), (w, 0), (w, h // 2), (0, h // 2))])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200, help="timed steps per path (split over the rounds)")
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--streams", type=int, default=64)
    ap.add_argument("--profile-steps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("region_bench needs a GPU")
    dev = torch.device("cuda:0")
    blob_dir = os.environ.get("AICAM_BLOB_DIR") or os.path.join(os.environ.get("TMPDIR", "/tmp"), "aicam_region_blobs")
    yolo, reid = synth.make_blobs(blob_dir)
    bias = synth.shifted_class_bias(yolo)
    S, T = args.streams, 8
    video = synth.SynthVideo(S, (1080, 1920), n_frames=T, seed=7)

    def make(settings):
        p = TrackingPipeline(yolo, reid, S, device=dev, max_frame_hw=(1080, 1920),
                             stream_settings=[settings] * S if settings else None)
        synth.apply_class_bias(p.detector.engine, bias)
        p.tracker.count_stats = True
        return p

    pipes = {"a_off": make(None), "b_pass_all": make(pass_all()), "c_exclude_top_half": make(top_half())}
    for t in range(args.warmup):
        for p in pipes.values():
            p.step(list(video.frames(t)))
    stream = torch.cuda.Stream()
    graphs = {}
    for name, p in pipes.items():
        p.reset_streams(range(S))
        torch.cuda.synchronize()
        stream.wait_stream(torch.cuda.current_stream())
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=stream):
            p.step_table()
        torch.cuda.synchronize()
        graphs[name] = g
        p.tracker.crop_total.zero_()
        p.tracker.track_total.zero_()

    per_round = max(1, args.steps // args.rounds)
    times = {k: [] for k in pipes}
    step0 = 0
    for r in range(args.rounds):
        for name, p in pipes.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for i in range(per_round):
                p.frame_table.set(list(video.frames(step0 + i)))
                graphs[name].replay()
            e1.record()
            torch.cuda.synchronize()
            times[name].append(e0.elapsed_time(e1) / per_round)
        step0 += per_round
    steps = per_round * args.rounds
    a, b = (pipes[k].tracker for k in ("a_off", "b_pass_all"))
    same = all(torch.equal(x, y) for x, y in ((a.out_tracks, b.out_tracks), (a.out_conf, b.out_conf),
                                              (a.out_count, b.out_count), (a.track_total, b.track_total),
                                              (a.crop_total, b.crop_total)))
    res = {"benchmark": "region_step", "frame": "1080x1920", "streams": S, "graphed_list_steps": True,
           "regions_b": "pass-all: 1 include + 7 excludes x 32 vertices per stream",
           "regions_c": "exclude the top half of every frame", "steps_per_path": steps, "rounds": args.rounds, **card()}
    med = {}
    for name, p in pipes.items():
        med[name] = float(np.median(times[name]))
        res[name] = {"ms_per_step": round(med[name], 3), "ms_per_round": [round(x, 3) for x in times[name]],
                     "crops_per_step": round(int(p.tracker.crop_total.item()) / steps, 1),
                     "tracks_per_step": round(int(p.tracker.track_total.item()) / steps, 2),
                     "launches_per_step": p.launches_per_step(True)}
    res["b_minus_a_ms"] = round(med["b_pass_all"] - med["a_off"], 4)
    res["c_minus_a_ms"] = round(med["c_exclude_top_half"] - med["a_off"], 4)
    res["round_spread"] = {k: round(max(v) / min(v), 4) for k, v in times.items()}
    res["a_b_outputs_identical"] = bool(same)
    # region_kernel and filter_kernel alone: eager (b) steps under the profiler
    from torch.profiler import ProfilerActivity, profile
    pb = pipes["b_pass_all"]
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(args.profile_steps):
            pb.step(list(video.frames(i)))
        torch.cuda.synchronize()
    dets = int(pb.detector.num_dets.sum().item())
    kernels = {}
    for e in prof.key_averages():
        for k in ("region_kernel", "filter_kernel"):
            if k in e.key:
                kernels[k] = {"calls": e.count, "us_per_call": round(e.device_time_total / max(1, e.count), 2)}
    res["kernels_b"] = kernels
    res["kernels_b_detections_last_step"] = dets
    res["kernels_b_edge_tests_last_step"] = dets * 8 * 32
    print(json.dumps(res))


if __name__ == "__main__":
    main()
