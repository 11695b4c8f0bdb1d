"""Streams of different frame sizes, pitches and surface formats in one batched step: the frame table
(aicam_frame_table_*), K1 / detect / K5 over it, TrackingPipeline.step(list) and the frame loop (-m gpu).
Every comparison is bit-exact."""
import ctypes as C
import json
import os

import numpy as np
import pytest
import torch

from scenarios import LETTERBOX_SIZES, synth_image

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


class Table:
    """A frame table set from entries: a BGR [H, W, 3] / NV12 [H*3/2, W] tensor, or (luma [H, W], chroma [H/2, W])
    for an NV12 frame whose planes are separate allocations."""

    def __init__(self, entries, bound=(2160, 3840)):
        from ai_camera_b200 import _lib as L
        self.handle = C.c_void_p()
        _check(_lib().aicam_frame_table_create(0, len(entries), bound[0], bound[1], C.byref(self.handle)))
        descs = (L.FrameDesc * len(entries))()
        for d, e in zip(descs, entries):
            if isinstance(e, tuple):
                y, c = e
                d.data, d.chroma, d.h, d.w, d.pitch, d.kind = y.data_ptr(), c.data_ptr(), y.shape[0], y.shape[1], y.stride(0), 1
            elif e.dim() == 3:
                d.data, d.chroma, d.h, d.w, d.pitch, d.kind = e.data_ptr(), None, e.shape[0], e.shape[1], e.stride(0), 0
            else:
                h = e.shape[0] * 2 // 3
                d.data, d.chroma, d.h, d.w, d.pitch, d.kind = e.data_ptr(), e.data_ptr() + h * e.stride(0), h, e.shape[1], e.stride(0), 1
        _check(_lib().aicam_frame_table_set(self.handle, descs, len(entries), None))
        self.entries, self.n = entries, len(entries)

    def close(self):
        _lib().aicam_frame_table_destroy(self.handle)


def bgr(rng, h, w):
    return torch.from_numpy(synth_image(rng, h, w)).to(DEV)


def nv12(frame_bgr):
    from ai_camera_b200 import synth
    return synth.bgr_to_nv12(frame_bgr[None])[0].contiguous()


def to_bgr(entry):
    """The BGR frame an entry stands for (NV12 converted as aicam_nv12_to_bgr / cv2 do), contiguous."""
    if isinstance(entry, tuple):
        entry = torch.cat(entry, 0)
    if entry.dim() == 3:
        return entry.contiguous()
    h, w = entry.shape[0] * 2 // 3, entry.shape[1]
    out = torch.empty((1, h, w, 3), dtype=torch.uint8, device=DEV)
    _check(_lib().aicam_nv12_to_bgr(entry.contiguous().data_ptr(), 1, h, w, out.data_ptr(), None))
    return out[0]


def pitched(frame, extra):
    """A view of `frame` inside a larger surface: rows `extra` bytes longer than the frame's."""
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


def k1_table(table, fmt):
    out = torch.empty(table.n * K1_BYTES[fmt], dtype=torch.uint8, device=DEV)
    _check(_lib().aicam_preprocess_table(table.handle, fmt, out.data_ptr(), None))
    return out.view(table.n, -1)


def test_k1_table_equals_uniform_entry_per_frame():
    rng = np.random.default_rng(3)
    entries = [bgr(rng, h, w) for h, w in LETTERBOX_SIZES + [(2160, 3840)]]
    entries += [nv12(bgr(rng, h, w)) for h, w in LETTERBOX_SIZES if h % 2 == 0 and w % 2 == 0]
    assert any(e.dim() == 3 and tuple(e.shape[:2]) == (1080, 1920) for e in entries)  # row-staged and per-pixel in one call
    t = Table(entries)
    try:
        for fmt in range(4):
            got = k1_table(t, fmt)
            for i, e in enumerate(entries):
                assert torch.equal(got[i], k1_uniform(e, fmt)), (fmt, i, tuple(e.shape))
    finally:
        t.close()


@pytest.mark.parametrize("bound", [(1080, 1930), (1080, 16000)])
def test_k1_table_with_unaligned_or_wide_bound(bound):
    """A width bound whose BGR row is not a multiple of 16 bytes (the ring's row slots are rounded up), and one so wide that
    the format-3 ring would not fit in shared memory (every frame then takes the per-pixel path)."""
    rng = np.random.default_rng(4)
    entries = [bgr(rng, 1080, 1920), bgr(rng, 480, 640), nv12(bgr(rng, 1080, 1920)), bgr(rng, 540, 960)]
    t = Table(entries, bound=bound)
    try:
        for fmt in range(4):
            got = k1_table(t, fmt)
            for i, e in enumerate(entries):
                assert torch.equal(got[i], k1_uniform(e, fmt)), (fmt, i)
    finally:
        t.close()


@pytest.mark.parametrize("kind", ["bgr", "nv12"])
def test_k1_uniform_table_equals_stacked_entry(kind):
    gen = torch.Generator(device=DEV).manual_seed(5)
    B, H, W = 64, 1080, 1920
    shape = (B, H, W, 3) if kind == "bgr" else (B, H * 3 // 2, W)
    frames = torch.randint(0, 256, shape, dtype=torch.uint8, device=DEV, generator=gen)
    want = torch.empty(B * K1_BYTES[3], dtype=torch.uint8, device=DEV)
    fn = _lib().aicam_preprocess if kind == "bgr" else _lib().aicam_preprocess_nv12
    _check(fn(frames.data_ptr(), B, H, W, 3, want.data_ptr(), None))
    t = Table(list(frames), bound=(1080, 1920))
    try:
        assert torch.equal(k1_table(t, 3).flatten(), want)
    finally:
        t.close()


def _boxes_for(sizes, rng, K=24):
    """[n, K, 4] boxes, scores, labels, num: random person-sized boxes plus ones that touch each frame's last row and column."""
    n = len(sizes)
    boxes = np.zeros((n, K, 4), np.float32)
    for b, (h, w) in enumerate(sizes):
        boxes[b, 0] = (w - 40.5, h - 90.2, w + 5.0, h + 3.0)
        boxes[b, 1] = (0, 0, w, h)
        boxes[b, 2] = (w - 1.5, 0.2, w + 0.0, h - 0.1)
        for k in range(3, K):
            x, y = rng.uniform(-20, w), rng.uniform(-20, h)
            boxes[b, k] = (x, y, x + rng.uniform(2, 0.4 * w + 3), y + rng.uniform(2, 0.6 * h + 3))
    scores = rng.choice(np.float32([0.2, 0.9, 0.5]), (n, K)).astype(np.float32)
    labels = rng.choice(np.int32([0, 2, 1, 7]), (n, K)).astype(np.int32)
    num = rng.integers(K // 2, K + 1, n).astype(np.int32)
    return [torch.from_numpy(a).to(DEV) for a in (boxes, scores, labels, num)]


def k5(table_or_frame, dets, fmt=0, max_crops=None):
    """aicam_reid_crops_table (a Table) or aicam_reid_crops[_nv12] (one frame entry, batch 1) -> numpy outputs."""
    from ai_camera_b200.config import tracked_class_mask
    boxes, scores, labels, num = dets
    B, K = scores.shape
    cap = max_crops or B * K
    o = dict(det_index=torch.full((B, K), -7, dtype=torch.int32, device=DEV), det_count=torch.zeros(B, dtype=torch.int32, device=DEV),
             crop_slot=torch.full((B, K), -7, dtype=torch.int32, device=DEV), crop_rect=torch.zeros((cap, 5), dtype=torch.int32, device=DEV),
             crops=torch.zeros((cap, 3, 128, 64) if fmt == 0 else (cap, 128, 64, 8), dtype=torch.float32 if fmt == 0 else torch.bfloat16, device=DEV),
             crop_count=torch.zeros(2, dtype=torch.int32, device=DEV))
    lo, hi = tracked_class_mask()
    tail = (boxes.data_ptr(), scores.data_ptr(), labels.data_ptr(), num.data_ptr(), K, 0.3, lo, hi, fmt, cap,
            o["det_index"].data_ptr(), o["det_count"].data_ptr(), o["crop_slot"].data_ptr(), o["crop_rect"].data_ptr(),
            o["crops"].data_ptr(), o["crop_count"].data_ptr(), None)
    if isinstance(table_or_frame, Table):
        _check(_lib().aicam_reid_crops_table(table_or_frame.handle, *tail))
    else:
        f = table_or_frame.contiguous() if not isinstance(table_or_frame, tuple) else torch.cat(table_or_frame, 0)
        if f.dim() == 3:
            _check(_lib().aicam_reid_crops(f.data_ptr(), 1, f.shape[0], f.shape[1], *tail))
        else:
            _check(_lib().aicam_reid_crops_nv12(f.data_ptr(), 1, f.shape[0] * 2 // 3, f.shape[1], *tail))
    torch.cuda.synchronize()
    out = {k: v.cpu() for k, v in o.items()}
    out["n"] = int(out["crop_count"][0])
    return out


def _frame_hw(e):
    if isinstance(e, tuple):
        return tuple(e[0].shape)
    return tuple(e.shape[:2]) if e.dim() == 3 else (e.shape[0] * 2 // 3, e.shape[1])


def test_k5_table_equals_per_frame_calls_and_oracle():
    from oracle import image_ops
    rng = np.random.default_rng(11)
    # 101 x 37 BGR: 11 211 bytes, not a multiple of 4 - its crops must not load whole words past its end
    entries = [bgr(rng, 540, 960), nv12(bgr(rng, 480, 640)), bgr(rng, 101, 37), nv12(bgr(rng, 300, 500)),
               bgr(rng, 1080, 1920), bgr(rng, 719, 1283)]
    sizes = [_frame_hw(e) for e in entries]
    dets = _boxes_for(sizes, rng)
    t = Table(entries)
    try:
        got = k5(t, dets)
    finally:
        t.close()
    base, checked = 0, 0
    for b, e in enumerate(entries):
        one = k5(e, [d[b:b + 1] for d in dets])
        nb = int(one["det_count"][0])
        assert int(got["det_count"][b]) == nb
        assert torch.equal(got["det_index"][b, :nb], one["det_index"][0, :nb])
        slots = one["crop_slot"][0, :nb]
        assert torch.equal(got["crop_slot"][b, :nb], torch.where(slots >= 0, slots + base, slots)), b
        frame = to_bgr(e).cpu().numpy()
        for k in range(one["n"]):
            r = got["crop_rect"][base + k].tolist()
            assert r[0] == b and r[1:] == one["crop_rect"][k, 1:].tolist()
            assert torch.equal(got["crops"][base + k], one["crops"][k])
            want = image_ops.preprocess_reid_input(frame[r[2]:r[4], r[1]:r[3]])
            assert np.array_equal(got["crops"][base + k].numpy(), np.asarray(want).reshape(3, 128, 64)), (b, k)
            checked += 1
        base += one["n"]
    assert got["n"] == base and checked > 20
    # the boxes at the last row / column of the 101 x 37 frame produced crops
    assert (got["crop_rect"][:base, 0] == 2).sum() > 0


@pytest.fixture(scope="module")
def blobs(tmp_path_factory):
    from ai_camera_b200 import synth
    return synth.make_blobs(str(tmp_path_factory.mktemp("blobs")))


def _video_frame(h, w, seed, t=0, n_frames=1):
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
        f = table_or_frame.contiguous() if not isinstance(table_or_frame, tuple) else torch.cat(table_or_frame, 0)
        out = det.detect(f[None])
    torch.cuda.synchronize()
    return [o.cpu() for o in out]


def test_detect_table_unletterboxes_per_frame(blobs):
    yolo, _ = blobs
    sizes = [(1080, 1920), (540, 960), (720, 1280), (2160, 3840), (480, 640), (641, 1283)]
    entries = [_video_frame(h, w, 40 + i)[0] for i, (h, w) in enumerate(sizes)]
    entries[2] = nv12(entries[2])
    det = _detector(yolo, len(entries), -0.6)
    t = Table(entries)
    try:
        got = _detect_host(det, t)
    finally:
        t.close()
    with_dets = 0
    for b, e in enumerate(entries):
        one = _detect_host(det, e)
        n = int(one[0][0])
        assert int(got[0][b]) == n, b
        for g, o in zip(got[1:], one[1:]):
            assert torch.equal(g[b], o[0]), b
        with_dets += n > 0
    assert with_dets >= len(entries) - 1, "too few frames with detections"


def test_pitched_frames_equal_contiguous_copies(blobs):
    yolo, _ = blobs
    rng = np.random.default_rng(21)
    base = [_video_frame(1080, 1920, 50)[0], _video_frame(540, 960, 51)[0], _video_frame(720, 1280, 52)[0], nv12(_video_frame(540, 960, 53)[0])]
    views = [pitched(base[0], 32),    # pitch 5 792: a multiple of 16 (row-staged K1)
             pitched(base[1], 4),     # pitch 2 884: a multiple of 4 only
             pitched(base[2], 64),
             (pitched(base[3][:540], 16), pitched(base[3][540:], 16))]  # NV12 with its chroma plane a separate allocation
    assert views[0].stride(0) % 16 == 0 and views[1].stride(0) % 16 == 4
    tv, tc = Table(views), Table(base)
    try:
        for fmt in range(4):
            assert torch.equal(k1_table(tv, fmt), k1_table(tc, fmt)), fmt
        dets = _boxes_for([_frame_hw(e) for e in base], rng)
        a, b = k5(tv, dets, fmt=2), k5(tc, dets, fmt=2)
        assert a["n"] > 0
        for k in ("det_index", "det_count", "crop_slot", "crop_rect", "crops", "crop_count"):
            assert torch.equal(a[k], b[k]), k
        det = _detector(yolo, 4, -0.6)
        da, db = _detect_host(det, tv), _detect_host(det, tc)
        assert int(da[0].sum()) > 0
        for x, y in zip(da, db):
            assert torch.equal(x, y)
    finally:
        tv.close()
        tc.close()


def _rows(ot, oc, on, s):
    from ai_camera_b200 import config
    return [tuple(int(v) for v in ot[s, k, :5]) + (config.CLASSES[ot[s, k, 5]], float(oc[s, k])) for k in range(on[s])]


def test_pipeline_list_step_equals_single_stream_facades(blobs):
    """The acceptance test: five streams of different sizes (one NV12, one pitched) in one list step per time step give,
    per stream, exactly the tuples of the single-stream facades on the same frames."""
    from ai_camera_b200 import synth
    from ai_camera_b200.deepsort_tracker import DeepSORT
    from ai_camera_b200.pipeline import TrackingPipeline
    from ai_camera_b200.yolo_detector import YOLODetector
    yolo, reid = blobs
    sizes = [(540, 960), (720, 1280), (1080, 1920), (480, 640), (600, 800)]
    T = 6
    videos = [_video_frame(h, w, 60 + i, n_frames=T) for i, (h, w) in enumerate(sizes)]
    bias = synth.shifted_class_bias(yolo, -0.6)
    pipe = TrackingPipeline(yolo, reid, len(sizes), max_tracks=128, n_init=2)
    synth.apply_class_bias(pipe.detector.engine, bias)
    det = YOLODetector(yolo)
    synth.apply_class_bias(det.trt_engine, bias)
    trks = [DeepSORT(reid, n_init=2, max_dets=100, max_tracks=128) for _ in sizes]
    reported = 0
    for t in range(T):
        frames = [v[t] for v in videos]
        frames[3] = nv12(frames[3])
        frames[1] = pitched(frames[1], 48)
        ot, oc, on = pipe.step(frames)
        torch.cuda.synchronize()
        ot, oc, on = ot.cpu().numpy(), oc.cpu().numpy(), on.cpu().numpy()
        for s in range(len(sizes)):
            frame = to_bgr(frames[s]).cpu().numpy()
            b, sc, c, _ = det.detect(frame)
            want = trks[s].update(b, sc, c, frame)
            assert _rows(ot, oc, on, s) == want, (t, s)
            reported += len(want)
    assert reported > 0
    assert not pipe.tracker.overflow().any()


def test_list_of_equal_frames_equals_stacked_tensor(blobs):
    from ai_camera_b200 import synth
    from ai_camera_b200.pipeline import TrackingPipeline
    yolo, reid = blobs
    S = 64
    video = synth.SynthVideo(S, (1080, 1920), n_frames=4, seed=7)
    bias = synth.shifted_class_bias(yolo)
    pipes = [TrackingPipeline(yolo, reid, S, max_tracks=128) for _ in range(2)]
    for p in pipes:
        synth.apply_class_bias(p.detector.engine, bias)
    total = 0
    for t in range(4):
        a = [x.cpu().numpy() for x in pipes[0].step(list(video.frames(t)))]
        b = [x.cpu().numpy() for x in pipes[1].step(video.frames(t))]
        assert np.array_equal(a[2], b[2]), t
        for s in range(S):
            assert _rows(*a, s) == _rows(*b, s), (t, s)
        total += int(a[2].sum())
    assert total > 0
    # the list path launches one kernel more (K1's per-pixel launch, made whatever the sizes), as launches_per_step says
    lib = _lib()
    counts = []
    for p, frames in ((pipes[0], list(video.frames(0))), (pipes[1], video.frames(0))):
        before = lib.aicam_launch_count()
        p.step(frames)
        counts.append(lib.aicam_launch_count() - before)
    assert counts[0] - counts[1] == pipes[0].launches_per_step(True) - pipes[0].launches_per_step() == 1


def test_captured_list_step_follows_the_table(blobs):
    """A step captured once stays valid when the table is set to other frames of other sizes within the bound."""
    from ai_camera_b200 import synth
    from ai_camera_b200.pipeline import TrackingPipeline
    yolo, reid = blobs
    bias = synth.shifted_class_bias(yolo, -0.6)
    first = [_video_frame(h, w, 70 + i)[0] for i, (h, w) in enumerate([(540, 960), (1080, 1920), (480, 640)])]
    other = [_video_frame(h, w, 80 + i, n_frames=3) for i, (h, w) in enumerate([(1080, 1920), (720, 1280), (600, 800)])]
    steps = [[v[t] for v in other] for t in range(3)]
    for st in steps:
        st[2] = nv12(st[2])
    pipes = [TrackingPipeline(yolo, reid, 3, max_tracks=128, n_init=1, max_frame_hw=(1080, 1920)) for _ in range(2)]
    for p in pipes:
        synth.apply_class_bias(p.detector.engine, bias)
    g_pipe, e_pipe = pipes
    g_pipe.step(first)  # warm-up: geometry tables, kernel attributes
    torch.cuda.synchronize()
    g_pipe.tracker.reset()
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=stream):
        out = g_pipe.step_table()
    reported = 0
    for frames in steps:
        g_pipe.frame_table.set(frames)
        g.replay()
        want = e_pipe.step(frames)
        torch.cuda.synchronize()
        got = [x.cpu().numpy() for x in out]
        want = [x.cpu().numpy() for x in want]
        assert np.array_equal(got[2], want[2])
        for s in range(3):
            assert _rows(*got, s) == _rows(*want, s), s
        reported += int(want[2].sum())
    assert reported > 0


def test_frame_table_set_rejects_malformed_descriptors():
    from ai_camera_b200 import _lib as L
    lib = _lib()
    buf = torch.zeros(1 << 20, dtype=torch.uint8, device=DEV)
    h = C.c_void_p()
    _check(lib.aicam_frame_table_create(0, 2, 1080, 1920, C.byref(h)))
    p = buf.data_ptr()
    cases = [  # (data, chroma, h, w, pitch, kind), expected code
        ((None, None, 100, 100, 300, 0), -1),
        ((p, None, 100, 100, 400, 1), -1),           # NV12 without a chroma plane
        ((p, None, 0, 100, 300, 0), -1),
        ((p, None, 100, -4, 300, 0), -1),
        ((p, None, 1081, 100, 300, 0), -4),           # above the bound
        ((p, None, 100, 1921, 6000, 0), -4),
        ((p, p, 101, 100, 100, 1), -1),               # odd NV12 height
        ((p, p, 100, 99, 100, 1), -1),                # odd NV12 width
        ((p, None, 100, 100, 299, 0), -1),            # pitch < row bytes
        ((p, p, 100, 100, 99, 1), -1),
        ((p, None, 100, 100, 300, 2), -1),            # unknown kind
    ]
    try:
        for fields, code in cases:
            descs = (L.FrameDesc * 1)(L.FrameDesc(*fields))
            before = lib.aicam_launch_count()
            assert lib.aicam_frame_table_set(h, descs, 1, None) == code, fields
            assert lib.aicam_launch_count() == before
        ok = (L.FrameDesc * 3)(*[L.FrameDesc(p, None, 100, 100, 300, 0)] * 3)
        before = lib.aicam_launch_count()
        assert lib.aicam_frame_table_set(h, ok, 3, None) == -4  # n > capacity
        assert lib.aicam_frame_table_set(h, ok, 2, None) == 0
        assert lib.aicam_launch_count() == before
    finally:
        lib.aicam_frame_table_destroy(h)


def test_frame_table_rejects_a_view_whose_last_pitch_leaves_its_storage():
    from ai_camera_b200 import _lib as L
    from ai_camera_b200.pipeline import FrameTable
    t = FrameTable(DEV, 2, (1080, 1920))
    surface = torch.zeros((100, 3 * 200 + 64), dtype=torch.uint8, device=DEV)
    inside = surface[:, :3 * 200].view(100, 200, 3)                 # rows * pitch = the whole surface
    right = surface[:, 64:].view(100, 200, 3)                       # the last row's pitch would run 64 bytes past the end
    t.set([inside])
    with pytest.raises(L.AicamError):
        t.set([inside, right])


def test_frame_loop_runs_sources_of_different_sizes(blobs, tmp_path):
    import cv2
    from ai_camera_b200 import synth
    from ai_camera_b200.aicamera_tracker import main, run_batched, run_single_stream, tracks_to_rows, video_frames
    from ai_camera_b200.deepsort_tracker import DeepSORT
    from ai_camera_b200.pipeline import TrackingPipeline
    from ai_camera_b200.yolo_detector import YOLODetector
    yolo, reid = blobs
    small = list(video_frames(CLIP, 20))
    large = [cv2.resize(f, (1280, 720)) for f in small]
    bias = synth.shifted_class_bias(yolo, synth.CLIP_LOGIT_SHIFT)
    pipe = TrackingPipeline(yolo, reid, 2, max_tracks=128, n_init=2)
    synth.apply_class_bias(pipe.detector.engine, bias)
    got = [[], []]

    def on_step(step, batch, table):
        tabs = [t.numpy() for t in table]
        for s in range(2):
            got[s].append(tracks_to_rows(tabs, s))
    run_batched([small, large], pipe, on_step)
    assert len(got[0]) == 20
    total = 0
    for s, frames in enumerate((small, large)):
        det = YOLODetector(yolo)
        synth.apply_class_bias(det.trt_engine, bias)
        trk = DeepSORT(reid, n_init=2, max_dets=100, max_tracks=128)
        want = []
        run_single_stream(frames, det, trk, on_frame=lambda i, f, d, tr: want.append(tr))
        assert got[s] == want, s
        total += sum(len(r) for r in want)
    assert total > 0
    # the command line with two files of different sizes
    paths = []
    for name, frames in (("a", small[:5]), ("b", large[:5])):
        path = str(tmp_path / (name + ".mp4"))
        w = cv2.VideoWriter(path, cv2.VideoWriter_fourcc(*"mp4v"), 10, (frames[0].shape[1], frames[0].shape[0]))
        for f in frames:
            w.write(f)
        w.release()
        paths.append(path)
    out = tmp_path / "out"
    assert main(["--input", paths[0], "--input", paths[1], "--streams", "2", "--max_frames", "5", "--output_dir", str(out),
                 "--output_filename", "mixed", "--yolo_engine", yolo, "--reid_engine", reid]) == 0
    lines = [json.loads(l) for l in open(out / "mixed.tracks.jsonl")]
    assert {l["stream"] for l in lines} == {0, 1} and len(lines) == 10
