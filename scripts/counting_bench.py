#!/usr/bin/env python
"""Cost of line and zone counting: 64 synthetic 1080p BGR streams (synth.SynthVideo, the detector calibrated with
synth.shifted_class_bias), graphed list steps (captured once, replayed after frame_table.set):
  (a) no counting;
  (b) counting on every stream at the maxima: 16 lines and 16 zones of 32 vertices each, all classes.
Paths are timed in alternating rounds in one process (CUDA events, median over rounds).  Then the counter kernel alone:
`--kernel-iters` launches of aicam_counter_step on (b)'s last step rows, bracketed by CUDA events.  One JSON line.
    python scripts/counting_bench.py [--steps N] [--rounds R] [--warmup W] [--kernel-iters K]"""
import argparse
import json
import math
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ai_camera_b200 import config, synth  # noqa: E402
from ai_camera_b200.pipeline import CountingLine, CountingZone, StreamCounting, TrackingPipeline  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = (x.strip() for x in q.split(","))
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # the numbers stand without it, but say so
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": "unknown (%s)" % e}


def max_geometry(s, w=1920, h=1080):
    """16 lines and 16 zones of 32 vertices (star-shaped polygons, so concave) spread over the frame."""
    rng = np.random.default_rng(1000 + s)
    every = set(config.CLASSES)
    lines = [CountingLine((int(rng.integers(0, w)), int(rng.integers(0, h))), (int(rng.integers(0, w)), int(rng.integers(0, h))),
                          classes=every) for _ in range(16)]
    zones = []
    for _ in range(16):
        cx, cy, r = int(rng.integers(200, w - 200)), int(rng.integers(200, h - 200)), int(rng.integers(80, 400))
        pts = [(cx + int(r * (0.5 + 0.5 * (k % 2)) * math.cos(2 * math.pi * k / 32)),
                cy + int(r * (0.5 + 0.5 * (k % 2)) * math.sin(2 * math.pi * k / 32))) for k in range(32)]
        zones.append(CountingZone(pts, classes=every))
    return StreamCounting(lines, zones)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200, help="timed steps per path (split over the rounds)")
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--streams", type=int, default=64)
    ap.add_argument("--kernel-iters", type=int, default=2000)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("counting_bench needs a GPU")
    dev = torch.device("cuda:0")
    blob_dir = os.environ.get("AICAM_BLOB_DIR") or os.path.join(os.environ.get("TMPDIR", "/tmp"), "aicam_counting_blobs")
    yolo, reid = synth.make_blobs(blob_dir)
    bias = synth.shifted_class_bias(yolo)
    S, T = args.streams, 8
    video = synth.SynthVideo(S, (1080, 1920), n_frames=T, seed=7)

    def make(counting):
        p = TrackingPipeline(yolo, reid, S, device=dev, max_frame_hw=(1080, 1920), counting=counting)
        synth.apply_class_bias(p.detector.engine, bias)
        p.tracker.count_stats = True
        return p

    pipes = {"a_off": make(None), "b_counting": make([max_geometry(s) for s in range(S)])}
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
    a, b = (pipes[k].tracker for k in ("a_off", "b_counting"))
    same = all(torch.equal(x, y) for x, y in ((a.out_tracks, b.out_tracks), (a.out_conf, b.out_conf),
                                              (a.out_count, b.out_count), (a.track_total, b.track_total)))
    res = {"benchmark": "counting_step", "frame": "1080x1920", "streams": S, "graphed_list_steps": True,
           "geometry_b": "16 lines + 16 zones x 32 vertices per stream, all classes", "steps_per_path": steps,
           "rounds": args.rounds, **card()}
    med = {}
    for name, p in pipes.items():
        med[name] = float(np.median(times[name]))
        res[name] = {"ms_per_step": round(med[name], 3), "ms_per_round": [round(x, 3) for x in times[name]],
                     "tracks_per_step": round(int(p.tracker.track_total.item()) / steps, 2)}
    res["b_minus_a_ms"] = round(med["b_counting"] - med["a_off"], 4)
    res["round_spread_a_b"] = [round(max(times[k]) / min(times[k]), 4) for k in pipes]
    res["tracker_outputs_identical"] = bool(same)
    pc = pipes["b_counting"]
    res["b_events_last_step"] = int(pc.counter.event_count.sum().item())
    res["b_overflow"] = bool(pc.counter.overflow().any())
    # the counter kernel alone, on the last step's rows (its state and counters keep changing; the work per launch is the
    # geometry test of every reported row, the same at every launch)
    tr = pc.tracker
    for _ in range(20):
        pc.counter.step(tr.out_tracks, tr.out_count, tr.row_slots, pc.frame_table.present_ptr)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(args.kernel_iters):
        pc.counter.step(tr.out_tracks, tr.out_count, tr.row_slots, pc.frame_table.present_ptr)
    e1.record()
    torch.cuda.synchronize()
    rows = int(tr.out_count.sum().item())
    res["counter_kernel"] = {"launches": args.kernel_iters, "us_per_launch": round(1e3 * e0.elapsed_time(e1) / args.kernel_iters, 2),
                             "rows_per_launch": rows,
                             "edge_and_line_tests_per_launch": rows * (16 + 16 * 32)}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
