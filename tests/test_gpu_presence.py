"""Streams that skip frames, end early and restart in one batched step: absent frames in the frame table
(aicam_frame_table_set_present), K1 / detect / K5 over the packed present frames, the tracker's presence mask and
per-stream reset, TrackingPipeline.step(list with None) and the frame loop's until / refill (-m gpu).
Every comparison is bit-exact."""
import ctypes as C
import json
import os

import numpy as np
import pytest
import torch

from scenarios import synth_image

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")
CLIP = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "aicamera_test_clip.mp4")
K1_BYTES = {0: 3 * 640 * 640 * 4, 1: 640 * 640 * 8, 2: 640 * 640 * 8, 3: 640 * 640 * 8}


def _lib():
    from ai_camera_b200 import _lib as L
    return L.load()


def _check(rc):
    from ai_camera_b200 import _lib as L
    L.check(rc)


def _desc(d, e):
    if e is None:
        d.data, d.chroma, d.h, d.w, d.pitch, d.kind = None, None, 0, 0, 0, 0
    elif isinstance(e, tuple):
        y, c = e
        d.data, d.chroma, d.h, d.w, d.pitch, d.kind = y.data_ptr(), c.data_ptr(), y.shape[0], y.shape[1], y.stride(0), 1
    elif e.dim() == 3:
        d.data, d.chroma, d.h, d.w, d.pitch, d.kind = e.data_ptr(), None, e.shape[0], e.shape[1], e.stride(0), 0
    else:
        h = e.shape[0] * 2 // 3
        d.data, d.chroma, d.h, d.w, d.pitch, d.kind = e.data_ptr(), e.data_ptr() + h * e.stride(0), h, e.shape[1], e.stride(0), 1


class Table:
    """A frame table set from entries (None = absent): a BGR [H, W, 3] / NV12 [H*3/2, W] tensor, or (luma, chroma)."""

    def __init__(self, entries, bound=(2160, 3840)):
        from ai_camera_b200 import _lib as L
        self.handle = C.c_void_p()
        _check(_lib().aicam_frame_table_create(0, len(entries), bound[0], bound[1], C.byref(self.handle)))
        descs = (L.FrameDesc * len(entries))()
        present = (C.c_uint8 * len(entries))(*[e is not None for e in entries])
        for d, e in zip(descs, entries):
            _desc(d, e)
        _check(_lib().aicam_frame_table_set_present(self.handle, descs, present, len(entries), None))
        self.entries, self.n = entries, len(entries)
        self.n_present = sum(e is not None for e in entries)

    def close(self):
        _lib().aicam_frame_table_destroy(self.handle)


def bgr(rng, h, w):
    return torch.from_numpy(synth_image(rng, h, w)).to(DEV)


def nv12(frame_bgr):
    from ai_camera_b200 import synth
    return synth.bgr_to_nv12(frame_bgr[None])[0].contiguous()


def to_bgr(entry):
    if isinstance(entry, tuple):
        entry = torch.cat(entry, 0)
    if entry.dim() == 3:
        return entry.contiguous()
    h, w = entry.shape[0] * 2 // 3, entry.shape[1]
    out = torch.empty((1, h, w, 3), dtype=torch.uint8, device=DEV)
    _check(_lib().aicam_nv12_to_bgr(entry.contiguous().data_ptr(), 1, h, w, out.data_ptr(), None))
    return out[0]


def pitched(frame, extra):
    rows, row = frame.shape[0], frame[0].numel()
    surface = torch.full((rows, row + extra), 77, dtype=torch.uint8, device=DEV)
    view = surface[:, :row].view(frame.shape)
    view.copy_(frame)
    return view


def k1_uniform(entry, fmt):
    out = torch.empty(K1_BYTES[fmt], dtype=torch.uint8, device=DEV)
    f = entry.contiguous() if not isinstance(entry, tuple) else torch.cat(entry, 0)
    if f.dim() == 3:
        _check(_lib().aicam_preprocess(f.data_ptr(), 1, f.shape[0], f.shape[1], fmt, out.data_ptr(), None))
    else:
        _check(_lib().aicam_preprocess_nv12(f.data_ptr(), 1, f.shape[0] * 2 // 3, f.shape[1], fmt, out.data_ptr(), None))
    return out


def _frame_hw(e):
    if isinstance(e, tuple):
        return tuple(e[0].shape)
    return tuple(e.shape[:2]) if e.dim() == 3 else (e.shape[0] * 2 // 3, e.shape[1])


def test_k1_writes_present_frames_packed():
    rng = np.random.default_rng(3)
    frames = [bgr(rng, 1080, 1920), bgr(rng, 540, 960), nv12(bgr(rng, 720, 1280)), pitched(bgr(rng, 1080, 1920), 32),
              bgr(rng, 641, 1283), nv12(bgr(rng, 1080, 1920)), pitched(bgr(rng, 480, 640), 4), bgr(rng, 2160, 3840)]
    present = [1, 0, 1, 1, 0, 1, 0, 1]
    entries = [f if p else None for f, p in zip(frames, present)]
    t = Table(entries)
    try:
        for fmt in range(4):
            out = torch.full((t.n * K1_BYTES[fmt],), 0xA5, dtype=torch.uint8, device=DEV)
            _check(_lib().aicam_preprocess_table(t.handle, fmt, out.data_ptr(), None))
            got = out.view(t.n, -1)
            slot = 0
            for i, e in enumerate(entries):
                if e is None:
                    continue
                assert torch.equal(got[slot], k1_uniform(e, fmt)), (fmt, i, slot)
                slot += 1
            assert slot == t.n_present
            assert bool((got[slot:] == 0xA5).all()), fmt  # slots past the present count are not written
    finally:
        t.close()


def _boxes_for(sizes, rng, K=24):
    n = len(sizes)
    boxes = np.zeros((n, K, 4), np.float32)
    for b, (h, w) in enumerate(sizes):
        boxes[b, 0] = (w - 40.5, h - 90.2, w + 5.0, h + 3.0)
        boxes[b, 1] = (0, 0, w, h)
        for k in range(2, K):
            x, y = rng.uniform(-20, w), rng.uniform(-20, h)
            boxes[b, k] = (x, y, x + rng.uniform(2, 0.4 * w + 3), y + rng.uniform(2, 0.6 * h + 3))
    scores = rng.choice(np.float32([0.2, 0.9, 0.5]), (n, K)).astype(np.float32)
    labels = rng.choice(np.int32([0, 2, 1, 7]), (n, K)).astype(np.int32)
    num = rng.integers(K // 2, K + 1, n).astype(np.int32)
    return [torch.from_numpy(a).to(DEV) for a in (boxes, scores, labels, num)]


def k5(table_or_frame, dets, fmt=2):
    from ai_camera_b200.config import tracked_class_mask
    boxes, scores, labels, num = dets
    B, K = scores.shape
    cap = B * K
    o = dict(det_index=torch.full((B, K), -7, dtype=torch.int32, device=DEV), det_count=torch.full((B,), -7, dtype=torch.int32, device=DEV),
             crop_slot=torch.full((B, K), -7, dtype=torch.int32, device=DEV), crop_rect=torch.zeros((cap, 5), dtype=torch.int32, device=DEV),
             crops=torch.zeros((cap, 128, 64, 8), dtype=torch.bfloat16, device=DEV),
             crop_count=torch.zeros(2, dtype=torch.int32, device=DEV))
    lo, hi = tracked_class_mask()
    tail = (boxes.data_ptr(), scores.data_ptr(), labels.data_ptr(), num.data_ptr(), K, 0.3, lo, hi, fmt, cap,
            o["det_index"].data_ptr(), o["det_count"].data_ptr(), o["crop_slot"].data_ptr(), o["crop_rect"].data_ptr(),
            o["crops"].data_ptr(), o["crop_count"].data_ptr(), None)
    if isinstance(table_or_frame, Table):
        _check(_lib().aicam_reid_crops_table(table_or_frame.handle, *tail))
    else:
        f = table_or_frame.contiguous()
        if f.dim() == 3:
            _check(_lib().aicam_reid_crops(f.data_ptr(), 1, f.shape[0], f.shape[1], *tail))
        else:
            _check(_lib().aicam_reid_crops_nv12(f.data_ptr(), 1, f.shape[0] * 2 // 3, f.shape[1], *tail))
    torch.cuda.synchronize()
    out = {k: v.cpu() for k, v in o.items()}
    out["n"] = int(out["crop_count"][0])
    return out


def test_k5_absent_frames_keep_no_detection():
    rng = np.random.default_rng(11)
    frames = [bgr(rng, 540, 960), nv12(bgr(rng, 480, 640)), bgr(rng, 101, 37), bgr(rng, 1080, 1920), bgr(rng, 719, 1283)]
    present = [1, 0, 1, 0, 1]
    entries = [f if p else None for f, p in zip(frames, present)]
    dets = _boxes_for([_frame_hw(f) for f in frames], rng)
    assert int(dets[3].min()) > 0  # every frame, absent ones included, claims detections
    t = Table(entries)
    try:
        got = k5(t, dets)
    finally:
        t.close()
    base = 0
    for b, e in enumerate(entries):
        if e is None:
            assert int(got["det_count"][b]) == 0, b
            continue
        one = k5(e, [d[b:b + 1] for d in dets])
        nb = int(one["det_count"][0])
        assert nb > 0 and int(got["det_count"][b]) == nb
        assert torch.equal(got["det_index"][b, :nb], one["det_index"][0, :nb])
        slots = one["crop_slot"][0, :nb]
        assert torch.equal(got["crop_slot"][b, :nb], torch.where(slots >= 0, slots + base, slots)), b
        for k in range(one["n"]):
            assert got["crop_rect"][base + k].tolist() == [b] + one["crop_rect"][k, 1:].tolist()
            assert torch.equal(got["crops"][base + k], one["crops"][k])
        base += one["n"]
    assert got["n"] == base and base > 0
    assert all(int(r[0]) not in (1, 3) for r in got["crop_rect"][:base])


@pytest.fixture(scope="module")
def blobs(tmp_path_factory):
    from ai_camera_b200 import synth
    return synth.make_blobs(str(tmp_path_factory.mktemp("blobs")))


def _video(h, w, seed, n_frames=1):
    from ai_camera_b200 import synth
    return synth.SynthVideo(1, (h, w), n_frames=n_frames, seed=seed).ring[:, 0]


def _detector(yolo, batch, shift):
    from ai_camera_b200 import synth
    from ai_camera_b200.pipeline import BatchDetector
    det = BatchDetector(yolo, batch)
    synth.apply_class_bias(det.engine, synth.shifted_class_bias(yolo, shift))
    return det


def _detect_host(det, table_or_frame):
    if isinstance(table_or_frame, Table):
        out = det.detect_table(table_or_frame)
    else:
        out = det.detect(table_or_frame.contiguous()[None])
    torch.cuda.synchronize()
    return [o.cpu().clone() for o in out]


def test_detect_runs_the_packed_present_frames(blobs):
    yolo, _ = blobs
    sizes = [(1080, 1920), (540, 960), (720, 1280), (2160, 3840), (480, 640), (641, 1283)]
    frames = [_video(h, w, 40 + i)[0] for i, (h, w) in enumerate(sizes)]
    frames[2] = nv12(frames[2])
    det = _detector(yolo, len(frames), -0.6)
    full = Table(frames)
    try:
        want = _detect_host(det, full)  # (also leaves every output row non-zero for the calls below)
    finally:
        full.close()
    assert int((want[0] > 0).sum()) >= len(frames) - 1
    for present in ([1, 0, 1, 1, 0, 1], [0, 0, 0, 0, 0, 1], [1, 1, 1, 1, 1, 0]):
        t = Table([f if p else None for f, p in zip(frames, present)])
        try:
            got = _detect_host(det, t)
        finally:
            t.close()
        for b, p in enumerate(present):
            if p:
                for g, w in zip(got, want):
                    assert torch.equal(g[b], w[b]), (present, b)
                one = _detect_host(det, frames[b]) if frames[b].dim() == 3 else None
                if one is not None:
                    for g, o in zip(got, one):
                        assert torch.equal(g[b], o[0]), (present, b)
            else:
                assert int(got[0][b]) == 0
                for g in got[1:]:
                    assert not bool(g[b].any()), (present, b)
    # every frame absent: the network launches over a count of zero and every row is empty
    t = Table([None] * len(frames))
    try:
        got = _detect_host(det, t)
    finally:
        t.close()
    for g in got:
        assert not bool(g.any())


def _rows(ot, oc, on, s):
    from ai_camera_b200 import config
    return [tuple(int(v) for v in ot[s, k, :5]) + (config.CLASSES[ot[s, k, 5]], float(oc[s, k])) for k in range(on[s])]


def _snapshot(pipe, s):
    ints, floats = pipe.tracker.snapshot(s)
    return ints.copy(), floats.view(np.uint32).copy()


def _facades(yolo, reid, n, bias):
    from ai_camera_b200 import synth
    from ai_camera_b200.deepsort_tracker import DeepSORT
    from ai_camera_b200.yolo_detector import YOLODetector
    det = YOLODetector(yolo)
    synth.apply_class_bias(det.trt_engine, bias)
    return det, [DeepSORT(reid, n_init=2, max_dets=100, max_tracks=128) for _ in range(n)]


def test_pipeline_with_absent_streams_equals_facades_on_present_frames(blobs):
    """Five streams of different sizes (one NV12, one pitched) with a fixed presence schedule: each stream's tuples at
    its present steps equal a facade pair run on its present frames only; an absent step reports 0 and leaves the
    stream's tracker state as it was, bit for bit."""
    from ai_camera_b200 import synth
    from ai_camera_b200.pipeline import TrackingPipeline
    yolo, reid = blobs
    sizes = [(540, 960), (720, 1280), (1080, 1920), (480, 640), (600, 800)]
    T = 10
    schedule = [[t % 2 == 0, t < 6, t >= 3, True, t not in (4, 7)] for t in range(T)]
    videos = [_video(h, w, 60 + i, n_frames=T) for i, (h, w) in enumerate(sizes)]
    bias = synth.shifted_class_bias(yolo, -0.6)
    pipe = TrackingPipeline(yolo, reid, len(sizes), max_tracks=128, n_init=2)
    synth.apply_class_bias(pipe.detector.engine, bias)
    det, trks = _facades(yolo, reid, len(sizes), bias)
    used = [0] * len(sizes)
    reported, absent_checked = 0, 0
    for t in range(T):
        frames = []
        for s in range(len(sizes)):
            if not schedule[t][s]:
                frames.append(None)
                continue
            f = videos[s][used[s]]
            used[s] += 1
            frames.append(nv12(f) if s == 3 else (pitched(f, 48) if s == 1 else f))
        before = {s: _snapshot(pipe, s) for s in range(len(sizes)) if frames[s] is None}
        ot, oc, on = [x.cpu().numpy() for x in pipe.step(frames)]
        for s in range(len(sizes)):
            if frames[s] is None:
                assert on[s] == 0, (t, s)
                after = _snapshot(pipe, s)
                assert all(np.array_equal(a, b) for a, b in zip(before[s], after)), (t, s)
                absent_checked += len(after[0]) > 0
                continue
            frame = to_bgr(frames[s]).cpu().numpy()
            b, sc, c, _ = det.detect(frame)
            want = trks[s].update(b, sc, c, frame)
            assert _rows(ot, oc, on, s) == want, (t, s)
            reported += len(want)
    assert reported > 0 and absent_checked > 0
    assert not pipe.tracker.overflow().any()


def test_reset_streams_gives_a_slot_a_fresh_tracker(blobs):
    from ai_camera_b200 import synth
    from ai_camera_b200.pipeline import TrackingPipeline
    yolo, reid = blobs
    sizes = [(540, 960), (720, 1280), (480, 640)]
    T, R, k = 8, 4, 1
    videos = [_video(h, w, 90 + i, n_frames=T) for i, (h, w) in enumerate(sizes)]
    new_src = _video(600, 800, 99, n_frames=T - R)
    bias = synth.shifted_class_bias(yolo, -0.6)
    pipe = TrackingPipeline(yolo, reid, len(sizes), max_tracks=128, n_init=2)
    synth.apply_class_bias(pipe.detector.engine, bias)
    det, trks = _facades(yolo, reid, len(sizes) + 1, bias)
    ids_after = []
    for t in range(T):
        if t == R:
            pipe.reset_streams([k])
        frames = [v[t] for v in videos]
        if t >= R:
            frames[k] = new_src[t - R]
        ot, oc, on = [x.cpu().numpy() for x in pipe.step(frames)]
        for s in range(len(sizes)):
            f = frames[s].cpu().numpy()
            trk = trks[-1] if (s == k and t >= R) else trks[s]  # a fresh facade for the new source
            b, sc, c, _ = det.detect(f)
            assert _rows(ot, oc, on, s) == trk.update(b, sc, c, f), (t, s)
            if s == k and t >= R:
                ids_after += [int(ot[s, j, 4]) for j in range(on[s])]
    assert ids_after and min(ids_after) == 1


def test_captured_step_follows_presence(blobs):
    from ai_camera_b200 import synth
    from ai_camera_b200.pipeline import TrackingPipeline
    yolo, reid = blobs
    bias = synth.shifted_class_bias(yolo, -0.6)
    first = [_video(h, w, 70 + i)[0] for i, (h, w) in enumerate([(540, 960), (1080, 1920), (480, 640)])]
    other = [_video(h, w, 80 + i, n_frames=6) for i, (h, w) in enumerate([(1080, 1920), (720, 1280), (600, 800)])]
    masks = [[1, 1, 1], [1, 0, 1], [0, 0, 0], [0, 1, 1], [1, 1, 0], [1, 1, 1]]
    steps = [[other[s][t] if masks[t][s] else None for s in range(3)] for t in range(6)]
    for st in steps:
        if st[2] is not None:
            st[2] = nv12(st[2])
    pipes = [TrackingPipeline(yolo, reid, 3, max_tracks=128, n_init=1, max_frame_hw=(1080, 1920)) for _ in range(2)]
    for p in pipes:
        synth.apply_class_bias(p.detector.engine, bias)
    g_pipe, e_pipe = pipes
    g_pipe.step(first)
    torch.cuda.synchronize()
    g_pipe.tracker.reset()
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=stream):
        out = g_pipe.step_table()
    reported = 0
    for t, frames in enumerate(steps):
        g_pipe.frame_table.set(frames)
        g.replay()
        want = e_pipe.step(frames)
        torch.cuda.synchronize()
        got = [x.cpu().numpy() for x in out]
        want = [x.cpu().numpy() for x in want]
        assert np.array_equal(got[2], want[2]), t
        for s in range(3):
            assert _rows(*got, s) == _rows(*want, s), (t, s)
            if not masks[t][s]:
                assert got[2][s] == 0
        reported += int(want[2].sum())
    assert reported > 0


def test_absent_frames_launch_nothing_more(blobs):
    from ai_camera_b200.pipeline import TrackingPipeline
    yolo, reid = blobs
    frames = [_video(h, w, 30 + i)[0] for i, (h, w) in enumerate([(540, 960), (720, 1280), (1080, 1920), (480, 640)])]
    pipe = TrackingPipeline(yolo, reid, 4, max_tracks=64)
    lib = _lib()
    counts = []
    for fr in (frames, [frames[0], None, frames[2], None], [None] * 4, frames):
        pipe.step(fr)  # (warm: the first sight of a size allocates its geometry)
        before = lib.aicam_launch_count()
        pipe.step(fr)
        counts.append(lib.aicam_launch_count() - before)
    torch.cuda.synchronize()
    assert len(set(counts)) == 1, counts


def test_set_present_validates_present_descriptors_only():
    from ai_camera_b200 import _lib as L
    lib = _lib()
    buf = torch.zeros(1 << 20, dtype=torch.uint8, device=DEV)
    h = C.c_void_p()
    _check(lib.aicam_frame_table_create(0, 3, 1080, 1920, C.byref(h)))
    p = buf.data_ptr()
    bad = [((None, None, 100, 100, 300, 0), -1), ((p, None, 100, 100, 400, 1), -1), ((p, None, 1081, 100, 300, 0), -4),
           ((p, None, 100, 100, 299, 0), -1), ((p, None, 100, 100, 300, 2), -1), ((p, p, 101, 100, 100, 1), -1)]
    good = L.FrameDesc(p, None, 100, 100, 300, 0)
    try:
        before = lib.aicam_launch_count()
        for fields, code in bad:
            descs = (L.FrameDesc * 3)(good, L.FrameDesc(*fields), good)
            # absent: the malformed descriptor is not read
            assert lib.aicam_frame_table_set_present(h, descs, (C.c_uint8 * 3)(1, 0, 1), 3, None) == 0, fields
            # present: rejected as aicam_frame_table_set rejects it
            assert lib.aicam_frame_table_set_present(h, descs, (C.c_uint8 * 3)(1, 1, 0), 3, None) == code, fields
            assert lib.aicam_frame_table_set(h, descs, 3, None) == code, fields
        nulls = (L.FrameDesc * 3)(L.FrameDesc(None, None, 0, 0, 0, 0), good, L.FrameDesc(None, None, 0, 0, 0, 0))
        assert lib.aicam_frame_table_set_present(h, nulls, (C.c_uint8 * 3)(0, 1, 0), 3, None) == 0
        assert lib.aicam_frame_table_set_present(h, None, (C.c_uint8 * 3)(0, 0, 0), 3, None) == 0
        assert lib.aicam_frame_table_set_present(h, None, (C.c_uint8 * 3)(0, 1, 0), 3, None) == -1
        assert lib.aicam_frame_table_set_present(h, nulls, None, 3, None) == -1  # NULL mask: every frame present
        assert lib.aicam_frame_table_set_present(h, nulls, (C.c_uint8 * 4)(0, 0, 0, 0), 4, None) == -4
        assert lib.aicam_launch_count() == before
        ptr = lib.aicam_frame_table_present(h)
        _check(lib.aicam_frame_table_set_present(h, nulls, (C.c_uint8 * 3)(0, 1, 0), 3, None))
        assert ptr and lib.aicam_frame_table_present(h) == ptr  # stable: a captured step reads it
        from ai_camera_b200.pipeline import FrameTable
        t = FrameTable(DEV, 3, (1080, 1920))
        t.set([None, buf[:300 * 100].view(100, 100, 3), None])
        torch.cuda.synchronize()
        assert t.n == 3 and t.n_present == 1
    finally:
        lib.aicam_frame_table_destroy(h)


def _write_clip(path, frames):
    import cv2
    w = cv2.VideoWriter(str(path), cv2.VideoWriter_fourcc(*"mp4v"), 10, (frames[0].shape[1], frames[0].shape[0]))
    for f in frames:
        w.write(f)
    w.release()
    return str(path)


def test_frame_loop_runs_every_input_to_its_end(blobs, tmp_path):
    import cv2
    from ai_camera_b200 import synth
    from ai_camera_b200.aicamera_tracker import main, run_batched, run_single_stream, tracks_to_rows, video_frames
    from ai_camera_b200.deepsort_tracker import DeepSORT
    from ai_camera_b200.pipeline import TrackingPipeline
    from ai_camera_b200.yolo_detector import YOLODetector
    yolo, reid = blobs
    clip = list(video_frames(CLIP, 20))
    inputs = [clip, [cv2.resize(f, (1280, 720)) for f in clip[:12]], [cv2.resize(f, (960, 540)) for f in clip[3:11]],
              clip[:15]]
    bias = synth.shifted_class_bias(yolo, synth.CLIP_LOGIT_SHIFT)
    pipe = TrackingPipeline(yolo, reid, 2, max_tracks=128, n_init=2)
    synth.apply_class_bias(pipe.detector.engine, bias)
    slot_input = [0, 1]
    got = [[] for _ in inputs]

    def on_refill(slot, k):
        slot_input[slot] = 2 + k

    def on_step(step, batch, table):
        tabs = [t.numpy() for t in table]
        for s, f in enumerate(batch):
            if f is not None:
                got[slot_input[s]].append(tracks_to_rows(tabs, s))
            else:
                assert int(tabs[2][s]) == 0
    run_batched(inputs[:2], pipe, on_step, until="all", refill=iter(inputs[2:]), on_refill=on_refill)
    total = 0
    for i, frames in enumerate(inputs):
        det = YOLODetector(yolo)
        synth.apply_class_bias(det.trt_engine, bias)
        trk = DeepSORT(reid, n_init=2, max_dets=100, max_tracks=128)
        want = []
        run_single_stream(frames, det, trk, on_frame=lambda i, f, d, tr: want.append(tr))
        assert got[i] == want, i
        total += sum(len(r) for r in want)
    assert total > 0
    # the command line: three inputs of different lengths through two slots
    lens = (5, 8, 3)
    paths = [_write_clip(tmp_path / ("%s.mp4" % n), fr) for n, fr in
             zip("abc", (clip[:lens[0]], [cv2.resize(f, (1280, 720)) for f in clip[:lens[1]]], clip[5:5 + lens[2]]))]
    out = tmp_path / "out"
    argv = sum((["--input", p] for p in paths), []) + ["--streams", "2", "--run_all_inputs", "--output_dir", str(out),
                                                     "--output_filename", "all", "--yolo_engine", yolo, "--reid_engine", reid]
    assert main(argv) == 0
    lines = [json.loads(l) for l in open(out / "all.tracks.jsonl")]
    for name, n in zip(("a.mp4", "b.mp4", "c.mp4"), lens):
        assert sorted(l["frame"] for l in lines if l["input"] == name) == list(range(n)), name
    assert len(lines) == sum(lens)
