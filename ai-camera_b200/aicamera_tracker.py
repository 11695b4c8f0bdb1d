"""The frame loop of the reference (``/root/reference/src/aicamera_tracker.py``) on the B200 path.

``python -m ai_camera_b200.aicamera_tracker --input clip.mp4 ...`` takes the reference's flags
(:20-67: ``--input --webcam_id --output_dir --output_filename --show_display --no_save
--yolo_engine --reid_engine --conf_thresh --device``) and runs its loop (:169-240): read a frame,
``YOLODetector.detect``, ``DeepSORT.update``, account the time the reference's way
(frames / sum of detect + update wall time, :175,199-207,254-258).

Differences, all in the direction of the hardware:
  * one frame upload per frame: ``detect`` leaves the frame in HBM and ``update`` is handed that
    device tensor (the reference passes ``frame_bgr.copy()`` through a second H2D inside its ReID
    preprocessing);
  * ``--streams N`` (new) runs N sources through ONE batched ``TrackingPipeline`` step per time
    step (the multi-camera form of the loop: per-stream order is kept, the N frames of a time
    step travel together; N = 1 keeps the reference-shaped facades);
  * the annotated video the reference writes (:211-236) is drawn ON THE DEVICE (visualization.py: box outlines,
    labels, status panel on a device copy of the frame the detector already uploaded) and only then copied back for
    ``cv2.VideoWriter`` (this image has no NVENC: the encode stays on the host); next to it the track tuples of every
    frame go to ``<stem>.tracks.jsonl``.  Batched mode writes videos only with ``--save_video`` (one per stream).
  * batched mode stops when its first input ends; ``--run_all_inputs`` (new) runs every input to its end instead: inputs
    beyond ``--streams`` wait for a slot whose input has ended, an ended slot without a waiting input is absent from
    the steps, track lines carry the input's name and ``--save_video`` writes one file per input.
  * ``--stream_settings FILE.json`` (new, batched mode) gives each input its own detection and tracking settings (the
    constructor arguments one reference process per input would take): ``{"default": {...}, "<input file name>": {...}}``
    with ``pipeline.StreamSettings`` field names.  An input's entry applies over "default", which applies over
    ``--conf_thresh`` and the config.  Each input runs with its entry from its first frame, also when it takes over a
    slot under ``--run_all_inputs``.
"""
import argparse
import json
import time
from pathlib import Path
from typing import Iterable, List, Optional

import numpy as np
import torch

from . import config


def parse_arguments(argv=None) -> argparse.Namespace:
    parser = argparse.ArgumentParser(description="AICamera: Real-time Object Detection & Tracking (B200 path)")
    parser.add_argument("--input", type=str, default=None, action="append",
                        help="Path to input video file (repeat for several streams). If None, tries to use webcam.")
    parser.add_argument("--webcam_id", type=int, default=0, help="Webcam ID to use if --input is not specified.")
    parser.add_argument("--output_dir", type=str, default="outputs", help="Directory to save the output.")
    parser.add_argument("--output_filename", type=str, default=None,
                        help="Name of the output file. If None, generated from input name or timestamp.")
    parser.add_argument("--show_display", action="store_true", help="Accepted for compatibility; no window is opened.")
    parser.add_argument("--no_save", action="store_true", help="Do not save the output video / track tables.")
    parser.add_argument("--save_video", action="store_true", help="Batched mode: also write one annotated video per stream.")
    parser.add_argument("--yolo_engine", type=str, default=str(config.YOLO_ENGINE_PATH),
                        help="Path to the YOLO weight blob (.aicw; replaces the TensorRT engine file).")
    parser.add_argument("--reid_engine", type=str, default=str(config.REID_ENGINE_PATH),
                        help="Path to the ReID (DeepSORT) weight blob (.aicw).")
    parser.add_argument("--conf_thresh", type=float, default=config.YOLO_CONF_THRESHOLD,
                        help="Confidence threshold for YOLO detections.")
    parser.add_argument("--device", type=str, default="cuda:0", help="CUDA device; there is no CPU path.")
    parser.add_argument("--streams", type=int, default=0,
                        help="Batched mode: number of streams per step (inputs are cycled to fill it). 0 = one "
                             "reference-shaped single-stream loop per input.")
    parser.add_argument("--max_frames", type=int, default=0, help="Stop after this many frames per stream (0 = all).")
    parser.add_argument("--run_all_inputs", action="store_true",
                        help="Batched mode: run every input to its end, whatever its length; inputs beyond --streams wait "
                             "for a free stream slot (a slot whose input has ended takes the next one with a fresh "
                             "tracker). Track lines carry the input's name and --save_video writes one file per input.")
    parser.add_argument("--stream_settings", type=str, default=None,
                        help="Batched mode: JSON file {\"default\": {...}, \"<input file name>\": {...}} of per-input "
                             "settings (conf_threshold, nms_threshold, classes_to_track, min_detection_confidence, "
                             "max_cosine_distance, max_iou_distance, max_age, n_init).")
    args = parser.parse_args(argv)
    if args.device == "cpu":
        parser.error("this build has no CPU path (the reference's TensorRT engines do not run on CPU either)")
    args.settings_for = None
    if args.stream_settings is not None:
        if args.streams <= 0:
            parser.error("--stream_settings needs batched mode (--streams N)")
        try:
            args.settings_for = load_stream_settings(args.stream_settings, args.conf_thresh)
        except (OSError, ValueError, TypeError) as e:
            parser.error("--stream_settings %s: %s" % (args.stream_settings, e))
    return args


def load_stream_settings(path, conf_threshold=config.YOLO_CONF_THRESHOLD):
    """The --stream_settings file as a function: input file name -> StreamSettings.  An input's entry applies over
    "default", which applies over ``conf_threshold`` and the config; an input without an entry gets "default"."""
    from .pipeline import StreamSettings
    with open(path) as f:
        spec = json.load(f)
    if not isinstance(spec, dict) or not all(isinstance(v, dict) for v in spec.values()):
        raise ValueError("expected a JSON object of objects")
    default = StreamSettings.from_dict(spec.get("default", {}), StreamSettings(conf_threshold=conf_threshold))
    entries = {name: StreamSettings.from_dict(v, default) for name, v in spec.items() if name != "default"}
    return lambda name: entries.get(name, default)


def input_name(spec):
    return Path(spec).name if isinstance(spec, str) else "webcam_%s" % spec


class LoopStats:
    """Timing as the reference accounts it (:175,199-207): per frame, wall time of detect + update."""

    def __init__(self):
        self.frame_ms: List[float] = []

    def add(self, seconds: float):
        self.frame_ms.append(1e3 * seconds)

    @property
    def frames(self):
        return len(self.frame_ms)

    @property
    def total_s(self):
        return sum(self.frame_ms) * 1e-3

    def fps(self):
        return self.frames / self.total_s if self.total_s > 0 else 0.0

    def percentile(self, q):
        return float(np.percentile(self.frame_ms, q)) if self.frame_ms else 0.0

    def summary(self):
        return {"frames": self.frames, "total_s": self.total_s, "avg_fps": self.fps(),
                "p50_ms": self.percentile(50), "p99_ms": self.percentile(99)}


def run_single_stream(frames: Iterable[np.ndarray], detector, tracker, on_frame=None, share_upload=True, stats_out=None) -> LoopStats:
    """The reference's while-loop body (:169-207) for one stream.  ``on_frame(idx, frame, dets, tracks)``
    receives what the loop would draw.  share_upload: hand ``update`` the frame ``detect`` already
    uploaded (one H2D per frame instead of two)."""
    stats = LoopStats()
    if stats_out is not None:
        stats_out.append(stats)  # (callbacks read the running fps from it)
    for idx, frame_bgr in enumerate(frames):
        t0 = time.time()
        det_bboxes, det_scores, det_class_ids, _ = detector.detect(frame_bgr)
        frame_arg = detector.device_frame if share_upload and detector.device_frame is not None else frame_bgr.copy()
        tracked = tracker.update(det_bboxes, det_scores, det_class_ids, frame_arg)
        stats.add(time.time() - t0)
        if on_frame is not None:
            on_frame(idx, frame_bgr, (det_bboxes, det_scores, det_class_ids), tracked)
    return stats


def run_batched(sources: List[Iterable[np.ndarray]], pipeline, on_step=None, max_steps=0, stats_out=None, until="first",
                refill: Optional[Iterable[Iterable[np.ndarray]]] = None, on_refill=None) -> LoopStats:
    """N streams, one ``TrackingPipeline.step`` per time step.  Frames are read on the host (cv2), staged in two
    pinned buffers and uploaded on a copy stream while the previous step computes; per-stream frame order is kept.
    Sources of different frame shapes get per-stream pinned and device buffers (two each) and the step takes the list
    of device frames.  Time per step = wall time from "frames of the step are on the host" to "track tables are on the
    host" (the detect + update span of the reference loop).

    until="first" (default): stop when the first source ends.  until="all": a source that has ended is absent from
    the steps that follow (None in ``batch`` for ``on_step``; it uploads nothing and its tracks are left as they are)
    and the loop ends when every source has ended.  refill: an iterable of further sources; a slot whose source ends
    takes the next one, after ``pipeline.reset_streams([slot])`` gave it a fresh tracker, and ``on_refill(slot, k)`` is
    told that it now holds refill source k (0-based).  With until="all" or a refill, every step takes the list of
    per-stream frames, and a slot's buffers are reallocated when its new source has another frame shape."""
    if until not in ("first", "all"):
        raise ValueError("until must be 'first' or 'all'")
    dev = pipeline.device
    its = [iter(s) for s in sources]
    S = pipeline.n_streams
    assert len(its) == S
    refill = iter(refill) if refill is not None else None
    n_refills = 0
    per_slot = until == "all" or refill is not None
    stats = LoopStats()
    if stats_out is not None:
        stats_out.append(stats)
    host = dev_buf = None
    T = pipeline.tracker.T
    out_host = [torch.empty((S, T, 6), dtype=torch.int32).pin_memory(), torch.empty((S, T), dtype=torch.float32).pin_memory(),
                torch.empty(S, dtype=torch.int32).pin_memory()]
    if per_slot:  # per slot and buffer parity: (pinned, device) staging of the slot's current frame shape
        host = [[None] * S for _ in range(2)]
        dev_buf = [[None] * S for _ in range(2)]
    step = 0
    while not max_steps or step < max_steps:
        batch = []
        for s in range(S):
            f = None
            while its[s] is not None:
                f = next(its[s], None)
                if f is not None:
                    break
                nxt = next(refill, None) if refill is not None else None
                if nxt is None:
                    if until == "first":
                        return stats
                    its[s] = None  # ended: absent from now on
                else:
                    its[s] = iter(nxt)
                    pipeline.reset_streams([s])
                    if on_refill is not None:
                        on_refill(s, n_refills)
                    n_refills += 1
            batch.append(f)
        if per_slot and all(f is None for f in batch):
            return stats
        if host is None:
            shapes = [tuple(f.shape) for f in batch]
            if all(sh == shapes[0] for sh in shapes):
                host = [torch.empty((S,) + shapes[0], dtype=torch.uint8).pin_memory() for _ in range(2)]
                dev_buf = [torch.empty((S,) + shapes[0], dtype=torch.uint8, device=dev) for _ in range(2)]
            else:  # one buffer per stream: the step takes the list of frames
                host = [[torch.empty(sh, dtype=torch.uint8).pin_memory() for sh in shapes] for _ in range(2)]
                dev_buf = [[torch.empty(sh, dtype=torch.uint8, device=dev) for sh in shapes] for _ in range(2)]
        h = host[step & 1]
        d = dev_buf[step & 1]
        if per_slot:
            for s, f in enumerate(batch):
                if f is not None and (h[s] is None or tuple(h[s].shape) != tuple(f.shape)):
                    h[s] = torch.empty(f.shape, dtype=torch.uint8).pin_memory()
                    d[s] = torch.empty(f.shape, dtype=torch.uint8, device=dev)
        for s, f in enumerate(batch):
            if f is not None:
                h[s].numpy()[...] = f
        t0 = time.time()
        if per_slot:
            frames_dev = []
            for s, f in enumerate(batch):
                if f is not None:
                    d[s].copy_(h[s], non_blocking=True)
                frames_dev.append(d[s] if f is not None else None)
            d = frames_dev
        elif isinstance(d, list):
            for ds, hs in zip(d, h):
                ds.copy_(hs, non_blocking=True)
        else:
            d.copy_(h, non_blocking=True)
        ot, oc, on = pipeline.step(d)
        out_host[0].copy_(ot, non_blocking=True)
        out_host[1].copy_(oc, non_blocking=True)
        out_host[2].copy_(on, non_blocking=True)
        torch.cuda.current_stream(dev).synchronize()
        stats.add(time.time() - t0)
        if on_step is not None:
            on_step(step, batch, out_host)
        step += 1
    return stats


def video_frames(path_or_id, max_frames=0):
    import cv2
    cap = cv2.VideoCapture(path_or_id)
    if not cap.isOpened():
        raise RuntimeError("Could not open video source (%s)." % path_or_id)
    n = 0
    try:
        while True:
            ok, frame = cap.read()
            if not ok:
                return
            yield frame
            n += 1
            if max_frames and n >= max_frames:
                return
    finally:
        cap.release()


class AnnotatedWriter:
    """The reference's visualisation + save step (:211-236) with the drawing on the device: ``write(frame_dev, tracks,
    lines)`` draws the tracks and the status panel on a device COPY of the frame (the reference draws on
    ``frame_bgr.copy()``), copies it back and hands it to cv2.VideoWriter (mp4v, as the reference :150-157)."""

    def __init__(self, path, device, fps=config.DEFAULT_OUTPUT_FPS):
        from .visualization import Overlay
        self.path, self.fps, self.device = str(path), fps, device
        self.overlay = Overlay(device)
        self.writer = None

    def write(self, frame_dev, tracked, info_lines):
        import cv2
        from .visualization import Overlay
        vis = frame_dev.reshape(frame_dev.shape[-3:]).clone()
        H, W = int(vis.shape[0]), int(vis.shape[1])
        lines = list(info_lines)
        self.overlay.draw(vis, [self.overlay.track_items(tracked, (H, W))],
                          panels=[(lambda img: Overlay._draw_info_panel(img, lines)) if lines else None])
        if self.writer is None:
            self.writer = cv2.VideoWriter(self.path, cv2.VideoWriter_fourcc(*"mp4v"), self.fps, (W, H))
            if not self.writer.isOpened():
                raise RuntimeError("Could not open video writer for %s" % self.path)
        self.writer.write(vis.cpu().numpy())

    def close(self):
        if self.writer is not None:
            self.writer.release()
            self.writer = None


def tracks_to_rows(table_host, s):
    ot, oc, on = table_host
    return [tuple(int(v) for v in ot[s, k, :5]) + (config.CLASSES[int(ot[s, k, 5])], float(oc[s, k])) for k in range(int(on[s]))]


def main(argv=None):
    args = parse_arguments(argv)
    device = torch.device(args.device)
    inputs = args.input or []
    for p in inputs:
        if not Path(p).exists():
            print(f"Error: Input video file not found: {p}")
            return 1
    names = [Path(p).stem for p in inputs] or [f"webcam_{args.webcam_id}"]
    sources_spec = inputs or [args.webcam_id]
    writer = None
    if not args.no_save:
        out_dir = Path(args.output_dir)
        out_dir.mkdir(parents=True, exist_ok=True)
        stem = Path(args.output_filename).stem if args.output_filename else "%s_tracked_%s" % (names[0], time.strftime("%Y%m%d-%H%M%S"))
        writer = open(out_dir / (stem + ".tracks.jsonl"), "w")
        print(f"Track tables will be saved to: {writer.name}")
    videos = []
    source_name = Path(inputs[0]).name if inputs else f"webcam_{args.webcam_id}"
    try:
        if args.streams > 0:
            from .pipeline import TrackingPipeline
            print("Initializing the batched pipeline (%d streams)..." % args.streams)
            stream_settings = None
            if args.settings_for:  # slot s starts with input s (inputs are cycled unless --run_all_inputs is given)
                first = [sources_spec[s % len(sources_spec)] if not args.run_all_inputs or s < len(sources_spec) else None
                         for s in range(args.streams)]
                stream_settings = [args.settings_for(input_name(p) if p is not None else None) for p in first]
            pipe = TrackingPipeline(args.yolo_engine, args.reid_engine, args.streams, device,
                                    conf_threshold=args.conf_thresh, stream_settings=stream_settings)
            if args.run_all_inputs:
                stats, frames = _run_all_inputs(args, pipe, sources_spec, writer, out_dir if writer else None,
                                                stem if writer else None, videos, device)
                return _summary(args, stats, frames)
            srcs = [video_frames(sources_spec[s % len(sources_spec)], args.max_frames) for s in range(args.streams)]

            if writer and args.save_video:
                videos = [AnnotatedWriter(out_dir / ("%s_s%02d.mp4" % (stem, s)), device) for s in range(args.streams)]
            dev_frames = {}
            pipe_step = pipe.step

            def step_and_keep(frames_dev, *a, **k):  # (the step's device frames, for the overlay)
                dev_frames["f"] = frames_dev
                return pipe_step(frames_dev, *a, **k)
            pipe.step = step_and_keep
            stats_ref = []

            def on_step(step, batch, table):
                if writer:
                    tabs = [t.numpy() for t in table]
                    fps = stats_ref[0].fps() * args.streams if stats_ref else 0.0
                    for s in range(args.streams):
                        rows = tracks_to_rows(tabs, s)
                        writer.write(json.dumps({"frame": step, "stream": s, "tracks": rows}) + "\n")
                        if videos:
                            videos[s].write(dev_frames["f"][s], rows, ["AICamera: YOLOv8 + DeepSORT", f"Input: {source_name}", "FPS: %.2f" % fps])
                if (step + 1) % 100 == 0:
                    print(f"Processed {step + 1} steps.")
            stats = run_batched(srcs, pipe, on_step, stats_out=stats_ref)
            frames = stats.frames * args.streams
        else:
            from .deepsort_tracker import DeepSORT
            from .yolo_detector import YOLODetector
            print("Initializing YOLOv8 Detector...")
            det = YOLODetector(engine_path=args.yolo_engine, conf_threshold=args.conf_thresh, device=device)
            print("Initializing DeepSORT Tracker...")
            trk = DeepSORT(reid_model_path=args.reid_engine, device=device)

            if writer:
                videos = [AnnotatedWriter(out_dir / (stem + ".mp4"), device)]
                print(f"Output video will be saved to: {videos[0].path}")
            loop_stats = []

            def on_frame(idx, frame, dets, tracks):
                if writer:
                    writer.write(json.dumps({"frame": idx, "stream": 0, "tracks": tracks}) + "\n")
                    fps = loop_stats[0].fps() if loop_stats else 0.0  # frames / sum of detect + update time, as the reference (:204-207)
                    videos[0].write(det.device_frame, tracks, ["AICamera: YOLOv8 + DeepSORT", f"Input: {source_name}", "FPS: %.2f" % fps])
                if (idx + 1) % 100 == 0:
                    print(f"Processed {idx + 1} frames.")
            stats = run_single_stream(video_frames(sources_spec[0], args.max_frames), det, trk, on_frame, stats_out=loop_stats)
            frames = stats.frames
    finally:
        if writer:
            writer.close()
        for v in videos:
            v.close()
    return _summary(args, stats, frames)


def _summary(args, stats, frames):
    print("\n--- Processing Summary ---")
    print(f"Total frames processed: {frames}")
    print(f"Total time: {stats.total_s:.2f} seconds")
    print(f"Average FPS: {frames / stats.total_s if stats.total_s > 0 else 0:.2f}")
    print("Latency per %s: p50 %.2f ms, p99 %.2f ms" % ("step" if args.streams > 0 else "frame", stats.percentile(50),
                                                        stats.percentile(99)))
    return 0


def _run_all_inputs(args, pipe, inputs, writer, out_dir, stem, videos, device):
    """--streams N --run_all_inputs: the first N inputs start in slots 0..N-1, the others wait for a slot whose input
    has ended; every input runs to its end (an ended slot without a waiting input is absent from the steps).  Returns
    (stats, frames processed)."""
    N = args.streams
    names = [input_name(p) for p in inputs]
    slot_input = [i if i < len(inputs) else None for i in range(N)]
    frame_idx = [0] * N
    srcs = [video_frames(inputs[i], args.max_frames) if i < len(inputs) else iter(()) for i in range(N)]
    refill = (video_frames(p, args.max_frames) for p in inputs[N:])
    if writer and args.save_video:
        videos.extend(AnnotatedWriter(out_dir / ("%s_in%02d_%s.mp4" % (stem, i, Path(n).stem)), device)
                      for i, n in enumerate(names))
    dev_frames = {}
    pipe_step = pipe.step

    def step_and_keep(frames_dev, *a, **k):  # (the step's device frames, for the overlay)
        dev_frames["f"] = frames_dev
        return pipe_step(frames_dev, *a, **k)
    pipe.step = step_and_keep
    stats_ref, counted = [], [0]

    def on_refill(slot, k):
        slot_input[slot] = N + k
        frame_idx[slot] = 0
        if args.settings_for:
            pipe.configure_streams([slot], args.settings_for(names[N + k]))

    def on_step(step, batch, table):
        tabs = [t.numpy() for t in table] if writer else None
        for s, f in enumerate(batch):
            if f is None:
                continue
            counted[0] += 1
            if writer:
                i = slot_input[s]
                rows = tracks_to_rows(tabs, s)
                writer.write(json.dumps({"frame": frame_idx[s], "stream": s, "input": names[i], "tracks": rows}) + "\n")
                if videos:
                    fps = stats_ref[0].fps() * N if stats_ref else 0.0
                    videos[i].write(dev_frames["f"][s], rows, ["AICamera: YOLOv8 + DeepSORT", f"Input: {names[i]}", "FPS: %.2f" % fps])
            frame_idx[s] += 1
        if (step + 1) % 100 == 0:
            print(f"Processed {step + 1} steps.")
    stats = run_batched(srcs, pipe, on_step, stats_out=stats_ref, until="all", refill=refill, on_refill=on_refill)
    return stats, counted[0]


if __name__ == "__main__":
    raise SystemExit(main())
