#!/usr/bin/env python
"""Whole-step benchmark of per-stream settings: 64 synthetic 1080p BGR streams (synth.SynthVideo, the detector calibrated
with synth.shifted_class_bias), graphed list steps (captured once, replayed after frame_table.set):
  (a) no per-stream settings;
  (b) every stream configured with settings equal to the constructor's (the per-entry and per-stream table path with
      neutral values): the same work as (a), its outputs must be identical;
  (c) four groups of 16 streams with different settings (vehicles only; people only at confidence 0.5; NMS IoU 0.4;
      max_age 10 with n_init 1): a different workload, reported with its ReID crops per step.
Paths are timed in alternating rounds in one process (CUDA events, median over rounds); one JSON line.
    python scripts/stream_settings_bench.py [--steps N] [--rounds R] [--warmup W]"""
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


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = (x.strip() for x in q.split(","))
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # the numbers stand without it, but say so
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": "unknown (%s)" % e}


GROUPS = [StreamSettings(classes_to_track={"car", "truck", "bus"}), StreamSettings(classes_to_track={"person"}, conf_threshold=0.5),
          StreamSettings(nms_threshold=0.4), StreamSettings(max_age=10, n_init=1)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200, help="timed steps per path (split over the rounds)")
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--streams", type=int, default=64)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("stream_settings_bench needs a GPU")
    dev = torch.device("cuda:0")
    blob_dir = os.environ.get("AICAM_BLOB_DIR") or os.path.join(os.environ.get("TMPDIR", "/tmp"), "aicam_settings_blobs")
    yolo, reid = synth.make_blobs(blob_dir)
    bias = synth.shifted_class_bias(yolo)
    S, T = args.streams, 8
    video = synth.SynthVideo(S, (1080, 1920), n_frames=T, seed=7)

    def make(settings):
        p = TrackingPipeline(yolo, reid, S, device=dev, max_frame_hw=(1080, 1920), stream_settings=settings)
        synth.apply_class_bias(p.detector.engine, bias)
        p.tracker.count_stats = True
        return p

    pipes = {"a_none": make(None), "b_neutral": make([StreamSettings()] * S),
             "c_four_groups": make([GROUPS[s * len(GROUPS) // S] for s in range(S)])}
    for t in range(args.warmup):
        for p in pipes.values():
            p.step(list(video.frames(t)))
    stream = torch.cuda.Stream()
    graphs = {}
    for name, p in pipes.items():
        p.tracker.reset()
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
    a, b = (pipes[k].tracker for k in ("a_none", "b_neutral"))
    same = all(torch.equal(x, y) for x, y in ((a.out_tracks, b.out_tracks), (a.out_conf, b.out_conf),
                                              (a.out_count, b.out_count), (a.crop_total, b.crop_total),
                                              (a.track_total, b.track_total)))
    res = {"benchmark": "stream_settings_step", "frame": "1080x1920", "streams": S, "graphed_list_steps": True,
           "steps_per_path": steps, "rounds": args.rounds, **card()}
    med = {}
    for name, p in pipes.items():
        med[name] = float(np.median(times[name]))
        res[name] = {"ms_per_step": round(med[name], 3), "ms_per_round": [round(x, 3) for x in times[name]],
                     "crops_per_step": round(int(p.tracker.crop_total.item()) / steps, 2),
                     "tracks_per_step": round(int(p.tracker.track_total.item()) / steps, 2)}
    res["b_over_a"] = round(med["b_neutral"] / med["a_none"], 4)
    spread = [max(times[k]) / min(times[k]) for k in ("a_none", "b_neutral")]
    res["round_spread_a_b"] = [round(x, 4) for x in spread]
    res["b_outputs_identical_to_a"] = bool(same)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
