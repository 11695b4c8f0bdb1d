#!/usr/bin/env python
"""Whole-step benchmark of streams of different frame sizes: one TrackingPipeline.step(list) per time step over a mixed
fleet of 16 x 2160x3840 + 16 x 1080x1920 + 16 x 720x1280 + 16 x 540x960 BGR streams (synth.SynthVideo per group, the
detector calibrated with synth.shifted_class_bias), eager and with the step captured once as a CUDA graph (the frame
table is set before every replay).  Next to it the uniform 64 x 1080p step through the list path and through the stacked
tensor path (eager, and graphed: one graph per ring position for the tensor path, whose graphs bake in the frame address).
Paths are timed in alternating rounds in one process (CUDA events, median over rounds); one JSON line.
    python scripts/ragged_bench.py [--steps N] [--rounds R] [--warmup W]"""
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

FLEET = [(2160, 3840), (1080, 1920), (720, 1280), (540, 960)]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = (x.strip() for x in q.split(","))
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # the numbers stand without it, but say so
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": "unknown (%s)" % e}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200, help="timed steps per path (split over the rounds)")
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--per_group", type=int, default=16)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    blob_dir = os.environ.get("AICAM_BLOB_DIR") or os.path.join(os.environ.get("TMPDIR", "/tmp"), "aicam_ragged_blobs")
    yolo, reid = synth.make_blobs(blob_dir)
    bias = synth.shifted_class_bias(yolo)
    G, T = args.per_group, 8
    groups = [synth.SynthVideo(G, hw, n_frames=T, seed=1000 + 97 * i) for i, hw in enumerate(FLEET)]
    uniform = synth.SynthVideo(4 * G, (1080, 1920), n_frames=T, seed=7)
    S = 4 * G

    def make():
        p = TrackingPipeline(yolo, reid, S, device=dev)
        synth.apply_class_bias(p.detector.engine, bias)
        p.tracker.count_stats = True
        return p

    def mixed_frames(t):
        return [f for g in groups for f in g.frames(t)]

    paths = {}
    # each path: (pipeline, step(t) callable)
    p_mixed = make()
    paths["mixed_eager"] = (p_mixed, lambda t: p_mixed.step(mixed_frames(t)))
    p_mixed_g = make()
    p_uni_list = make()
    paths["uniform_list_eager"] = (p_uni_list, lambda t: p_uni_list.step(list(uniform.frames(t))))
    p_uni_tensor = make()
    paths["uniform_tensor_eager"] = (p_uni_tensor, lambda t: p_uni_tensor.step(uniform.frames(t)))
    p_uni_list_g = make()
    p_uni_tensor_g = make()

    stream = torch.cuda.Stream()

    def capture(fn):
        torch.cuda.synchronize()
        stream.wait_stream(torch.cuda.current_stream())
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=stream):
            fn()
        torch.cuda.synchronize()
        return g

    # warm up every path eagerly (geometry tables, kernel attributes), then capture
    for t in range(args.warmup):
        for p, fn in paths.values():
            fn(t)
        p_mixed_g.step(mixed_frames(t))
        p_uni_list_g.step(list(uniform.frames(t)))
        p_uni_tensor_g.step(uniform.frames(t))
    torch.cuda.synchronize()
    g_mixed = capture(p_mixed_g.step_table)
    g_uni_list = capture(p_uni_list_g.step_table)
    tensor_graphs = [capture(lambda k=k: p_uni_tensor_g.step(uniform.ring[k])) for k in range(T)]

    def graphed_list(p, g, frames_of):
        def fn(t):
            p.frame_table.set(frames_of(t))
            g.replay()
        return fn
    paths["mixed_graph"] = (p_mixed_g, graphed_list(p_mixed_g, g_mixed, mixed_frames))
    paths["uniform_list_graph"] = (p_uni_list_g, graphed_list(p_uni_list_g, g_uni_list, lambda t: list(uniform.frames(t))))
    paths["uniform_tensor_graph"] = (p_uni_tensor_g, lambda t: tensor_graphs[uniform.index(t)].replay())
    for p, _ in paths.values():
        p.tracker.crop_total.zero_()
    per_round = max(1, args.steps // args.rounds)
    times = {k: [] for k in paths}
    step0 = args.warmup
    for r in range(args.rounds):
        for name, (p, fn) in paths.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for i in range(per_round):
                fn(step0 + i)
            e1.record()
            torch.cuda.synchronize()
            times[name].append(e0.elapsed_time(e1) / per_round)
        step0 += per_round
    total_steps = per_round * args.rounds
    res = {"benchmark": "ragged_step", "fleet": {"%dx%d" % hw: G for hw in FLEET}, "streams": S,
           "steps_per_path": total_steps, "rounds": args.rounds, **card()}
    for name, (p, _) in paths.items():
        ms = float(np.median(times[name]))
        res[name] = {"ms_per_step": round(ms, 3), "frames_per_s": round(S * 1e3 / ms, 1),
                     "ms_per_round": [round(x, 3) for x in times[name]],
                     "crops_per_step": round(float(p.tracker.crop_total.item()) / total_steps, 1)}
    res["uniform_list_over_tensor_eager"] = round(res["uniform_list_eager"]["ms_per_step"] / res["uniform_tensor_eager"]["ms_per_step"], 4)
    res["uniform_list_over_tensor_graph"] = round(res["uniform_list_graph"]["ms_per_step"] / res["uniform_tensor_graph"]["ms_per_step"], 4)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
