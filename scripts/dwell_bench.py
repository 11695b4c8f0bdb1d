#!/usr/bin/env python
"""Cost of dwell: 64 synthetic 1080p BGR streams (synth.SynthVideo, the detector calibrated with
synth.shifted_class_bias), graphed list steps (captured once, replayed after frame_table.set), counting at the maxima on
every stream (16 lines and 16 zones of 32 vertices each, all classes, as scripts/counting_bench.py):
  (a) dwell off;
  (b) dwell on every stream and zone, loiter thresholds of 1 to 16 frames so that alerts fire.
Paths are timed in alternating rounds in one process (CUDA events, median over rounds).  Then the dwell kernel alone:
`--kernel-iters` launches of aicam_counter_dwell_step on (b)'s last step rows, bracketed by CUDA events.  One JSON line.
    python scripts/dwell_bench.py [--steps N] [--rounds R] [--warmup W] [--kernel-iters K]"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ai_camera_b200 import synth  # noqa: E402
from ai_camera_b200.pipeline import TrackingPipeline  # noqa: E402

sys.path.insert(0, os.path.join(ROOT, "scripts"))
from counting_bench import card, max_geometry  # noqa: E402


def with_dwell(sc, s):
    """``sc`` with a loiter threshold of 1 to 16 frames on every zone."""
    from dataclasses import replace
    return replace(sc, zones=tuple(replace(z, loiter_frames=1 + (s + i) % 16) for i, z in enumerate(sc.zones)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200, help="timed steps per path (split over the rounds)")
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--streams", type=int, default=64)
    ap.add_argument("--kernel-iters", type=int, default=2000)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("dwell_bench needs a GPU")
    dev = torch.device("cuda:0")
    blob_dir = os.environ.get("AICAM_BLOB_DIR") or os.path.join(os.environ.get("TMPDIR", "/tmp"), "aicam_dwell_blobs")
    yolo, reid = synth.make_blobs(blob_dir)
    bias = synth.shifted_class_bias(yolo)
    S, T = args.streams, 8
    video = synth.SynthVideo(S, (1080, 1920), n_frames=T, seed=7)

    def make(counting):
        p = TrackingPipeline(yolo, reid, S, device=dev, max_frame_hw=(1080, 1920), counting=counting)
        synth.apply_class_bias(p.detector.engine, bias)
        p.tracker.count_stats = True
        return p

    geometry = [max_geometry(s) for s in range(S)]
    pipes = {"a_dwell_off": make(geometry), "b_dwell_on": make([with_dwell(g, s) for s, g in enumerate(geometry)])}
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
    pa, pb = pipes["a_dwell_off"], pipes["b_dwell_on"]
    a, b = pa.tracker, pb.tracker
    same = all(torch.equal(x, y) for x, y in ((a.out_tracks, b.out_tracks), (a.out_conf, b.out_conf),
                                              (a.out_count, b.out_count), (a.track_total, b.track_total)))
    same_counting = all(torch.equal(getattr(pa.counter, n), getattr(pb.counter, n))
                        for n in ("line_counts", "zone_counts", "occupancy", "row_zones", "events", "event_count"))
    res = {"benchmark": "dwell_step", "frame": "1080x1920", "streams": S, "graphed_list_steps": True,
           "counting": "16 lines + 16 zones x 32 vertices per stream, all classes",
           "dwell_b": "every stream and zone, loiter_frames 1..16", "steps_per_path": steps,
           "rounds": args.rounds, **card()}
    med = {}
    for name, p in pipes.items():
        med[name] = float(np.median(times[name]))
        res[name] = {"ms_per_step": round(med[name], 3), "ms_per_round": [round(x, 3) for x in times[name]],
                     "tracks_per_step": round(int(p.tracker.track_total.item()) / steps, 2),
                     "launches_per_step": p.launches_per_step(frame_list=True)}
    res["b_minus_a_ms"] = round(med["b_dwell_on"] - med["a_dwell_off"], 4)
    res["round_spread_a_b"] = [round(max(times[k]) / min(times[k]), 4) for k in pipes]
    res["tracker_outputs_identical"] = bool(same)
    res["counting_outputs_identical"] = bool(same_counting)
    res["b_dwell_events_last_step"] = int(pb.counter.dwell_event_count.sum().item())
    res["b_open_visits_last_step"] = int((pb.counter.row_dwell >= 0).sum().item())
    res["b_completed_visits"] = int(pb.counter.visits.sum().item())
    res["b_dwell_overflow"] = bool(pb.counter.dwell_overflow().any())
    # the dwell kernel alone, on the last step's rows (its clock, state and counters keep changing; the work per launch is
    # every reported row against every zone, the same at every launch)
    tr = pb.tracker
    for _ in range(20):
        pb.counter.dwell_step(tr.out_tracks, tr.out_count, tr.row_slots, pb.frame_table.present_ptr)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(args.kernel_iters):
        pb.counter.dwell_step(tr.out_tracks, tr.out_count, tr.row_slots, pb.frame_table.present_ptr)
    e1.record()
    torch.cuda.synchronize()
    rows = int(tr.out_count.sum().item())
    res["dwell_kernel"] = {"launches": args.kernel_iters, "us_per_launch": round(1e3 * e0.elapsed_time(e1) / args.kernel_iters, 2),
                           "rows_per_launch": rows, "row_zone_tests_per_launch": rows * 16}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
