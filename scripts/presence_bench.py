#!/usr/bin/env python
"""Whole-step benchmark of absent streams: what a step with some streams absent costs against a pipeline sized to the
present streams.  Synthetic 1080p BGR streams (synth.SynthVideo, the detector calibrated with synth.shifted_class_bias),
every step captured once as a CUDA graph and replayed after frame_table.set:
  (a) a 64-slot pipeline at 100 / 75 / 50 / 25 % presence, the absent set rotating every step;
  (b) per presence level, a pipeline of exactly the present count taking the same frames;
  (c) the all-present 64-stream list step against the stacked tensor step, eager and graphed (as scripts/ragged_bench.py).
Paths are timed in alternating rounds in one process (CUDA events, median over rounds); one JSON line.
    python scripts/presence_bench.py [--steps N] [--rounds R] [--warmup W]"""
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
from ai_camera_b200.pipeline import TrackingPipeline  # noqa: E402

LEVELS = (1.0, 0.75, 0.5, 0.25)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = (x.strip() for x in q.split(","))
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # the numbers stand without it, but say so
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": "unknown (%s)" % e}


def present_slots(S, n, t):
    """The n present slots of step t: a window that moves by S / 4 slots per step, so the absent set rotates."""
    off = (t * (S // 4)) % S
    return sorted((off + j) % S for j in range(n))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200, help="timed steps per path (split over the rounds)")
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--streams", type=int, default=64)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("presence_bench needs a GPU")
    dev = torch.device("cuda:0")
    blob_dir = os.environ.get("AICAM_BLOB_DIR") or os.path.join(os.environ.get("TMPDIR", "/tmp"), "aicam_presence_blobs")
    yolo, reid = synth.make_blobs(blob_dir)
    bias = synth.shifted_class_bias(yolo)
    S, T = args.streams, 8
    video = synth.SynthVideo(S, (1080, 1920), n_frames=T, seed=7)
    counts = {lv: int(round(S * lv)) for lv in LEVELS}

    def make(n):
        p = TrackingPipeline(yolo, reid, n, device=dev, max_frame_hw=(1080, 1920))
        synth.apply_class_bias(p.detector.engine, bias)
        return p

    def slot_frames(n, t):  # the 64-slot list: the present slots' frames, None elsewhere
        fr = list(video.frames(t))
        keep = set(present_slots(S, n, t))
        return [f if s in keep else None for s, f in enumerate(fr)]

    def packed_frames(n, t):  # the same frames for a pipeline of n streams
        fr = list(video.frames(t))
        return [fr[s] for s in present_slots(S, n, t)]

    stream = torch.cuda.Stream()

    def capture(fn):
        torch.cuda.synchronize()
        stream.wait_stream(torch.cuda.current_stream())
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=stream):
            fn()
        torch.cuda.synchronize()
        return g

    p_slots = make(S)
    p_sized = {n: make(n) for n in sorted(set(counts.values())) if n < S}
    p_sized[S] = p_slots  # all present: the sized pipeline is the 64-slot one
    p_list_e, p_tensor_e, p_tensor_g = make(S), make(S), make(S)
    for t in range(args.warmup):
        for n in counts.values():
            p_slots.step(slot_frames(n, t))
            p_sized[n].step(packed_frames(n, t))
        p_list_e.step(list(video.frames(t)))
        p_tensor_e.step(video.frames(t))
        p_tensor_g.step(video.frames(t))
    torch.cuda.synchronize()
    graphs = {n: capture(p.step_table) for n, p in p_sized.items()}
    tensor_graphs = [capture(lambda k=k: p_tensor_g.step(video.ring[k])) for k in range(T)]

    def graphed(p, n, frames_of):
        def fn(t):
            p.frame_table.set(frames_of(n, t))
            graphs[n if p is not p_slots else S].replay()
        return fn

    paths = {}
    for lv, n in counts.items():
        pct = int(round(100 * lv))
        paths["slots64_present%d" % pct] = graphed(p_slots, n, slot_frames)
        if n < S:
            paths["sized%d" % n] = graphed(p_sized[n], n, packed_frames)
    paths["uniform_list_eager"] = lambda t: p_list_e.step(list(video.frames(t)))
    paths["uniform_tensor_eager"] = lambda t: p_tensor_e.step(video.frames(t))
    paths["uniform_tensor_graph"] = lambda t: tensor_graphs[video.index(t)].replay()
    per_round = max(1, args.steps // args.rounds)
    times = {k: [] for k in paths}
    step0 = args.warmup
    for r in range(args.rounds):
        for name, fn in paths.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for i in range(per_round):
                fn(step0 + i)
            e1.record()
            torch.cuda.synchronize()
            times[name].append(e0.elapsed_time(e1) / per_round)
        step0 += per_round
    res = {"benchmark": "presence_step", "frame": "1080x1920", "slots": S, "steps_per_path": per_round * args.rounds,
           "rounds": args.rounds, **card()}
    med = {}
    for name in paths:
        med[name] = float(np.median(times[name]))
        res[name] = {"ms_per_step": round(med[name], 3), "ms_per_round": [round(x, 3) for x in times[name]]}
    for lv, n in counts.items():
        pct = int(round(100 * lv))
        if n < S:
            res["slots64_over_sized_present%d" % pct] = round(med["slots64_present%d" % pct] / med["sized%d" % n], 4)
    res["uniform_list_over_tensor_eager"] = round(med["uniform_list_eager"] / med["uniform_tensor_eager"], 4)
    # (the all-present 64-slot graph is the graphed list step)
    res["uniform_list_over_tensor_graph"] = round(med["slots64_present100"] / med["uniform_tensor_graph"], 4)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
