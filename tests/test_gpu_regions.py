"""Per-stream include and exclude regions on the device (aicam_frame_table_set_regions, region_kernel in K5): the crop
filter against oracle/regions.py and against a region-less run on host-compacted detections, tracking against a
region-less tracker fed the compacted detector outputs, the neutral and unchanged paths, routing, capture, resets, ABI
validation and the command line.  Everything is compared bit for bit."""
import ctypes as C
import json
import os
from dataclasses import replace

import numpy as np
import pytest
import torch

from oracle import regions as R
from scenarios import synth_image

DEV = torch.device("cuda:0")
CLIP = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "aicamera_test_clip.mp4")
LIMIT = 1 << 20
pytestmark = pytest.mark.gpu


def _L():
    from ai_camera_b200 import _lib as L
    return L


def _lib():
    return _L().load()


def _check(rc):
    _L().check(rc)


def _record(region):
    """aicam_stream_region of an oracle region (includes, excludes)."""
    r = _L().StreamRegion()
    polys = [(0, p) for p in region[0]] + [(1, p) for p in region[1]]
    r.n_polygons = len(polys)
    for i, (kind, pts) in enumerate(polys):
        r.kind[i], r.n_vertices[i] = kind, len(pts)
        for k, (x, y) in enumerate(pts):
            r.xy[i][k][:] = [x, y]
    return r


def _set_regions(handle, indices, records):
    n = len(indices)
    return _lib().aicam_frame_table_set_regions(handle, (C.c_int32 * n)(*indices), (_L().StreamRegion * n)(*records), n,
                                                None)


class Table:
    """A frame table set from entries (None = absent), with optional per-entry filters."""

    def __init__(self, entries, filters=None):
        L = _L()
        self.handle = C.c_void_p()
        _check(_lib().aicam_frame_table_create(0, len(entries), 2160, 3840, C.byref(self.handle)))
        if filters:
            _check(_lib().aicam_frame_table_set_filters(self.handle, (L.StreamFilter * len(filters))(*filters), len(filters)))
        self.descs = (L.FrameDesc * len(entries))()
        for d, e in zip(self.descs, entries):
            if e is None:
                continue
            if e.dim() == 3:
                d.data, d.chroma, d.h, d.w, d.pitch, d.kind = e.data_ptr(), None, e.shape[0], e.shape[1], e.stride(0), 0
            else:
                h = e.shape[0] * 2 // 3
                d.data, d.chroma, d.h, d.w, d.pitch, d.kind = (e.data_ptr(), e.data_ptr() + h * e.stride(0), h, e.shape[1],
                                                               e.stride(0), 1)
        self.present = (C.c_uint8 * len(entries))(*[e is not None for e in entries])
        self.n = len(entries)
        self.set()

    def set(self):
        _check(_lib().aicam_frame_table_set_present(self.handle, self.descs, self.present, self.n, None))

    def close(self):
        _lib().aicam_frame_table_destroy(self.handle)


def _filter(min_conf=0.3, classes=None):
    from ai_camera_b200 import config
    lo, hi = config.tracked_class_mask(classes)
    return _L().StreamFilter(0.3, 0.5, min_conf, 0, lo, hi)


def _k5(table, dets, K, cap, min_conf=0.3, mask=None):
    from ai_camera_b200 import config
    boxes, scores, labels, num = dets
    mask = mask or config.tracked_class_mask()
    B = num.shape[0]
    i32 = dict(dtype=torch.int32, device=DEV)
    o = dict(det_index=torch.full((B, K), -7, **i32), det_count=torch.full((B,), -7, **i32),
             crop_slot=torch.full((B, K), -7, **i32), crop_rect=torch.zeros((cap, 5), **i32),
             crops=torch.zeros((cap, 128, 64, 8), dtype=torch.bfloat16, device=DEV), crop_count=torch.zeros(2, **i32))
    rc = _lib().aicam_reid_crops_table(
        table.handle, boxes.data_ptr(), scores.data_ptr(), labels.data_ptr(), num.data_ptr(), K, min_conf, mask[0], mask[1],
        2, cap, o["det_index"].data_ptr(), o["det_count"].data_ptr(), o["crop_slot"].data_ptr(), o["crop_rect"].data_ptr(),
        o["crops"].data_ptr(), o["crop_count"].data_ptr(), None)
    _check(rc)
    torch.cuda.synchronize()
    out = {k: v.cpu() for k, v in o.items() if k != "crops"}
    out["crops"] = o["crops"][:int(out["crop_count"][0])].cpu()
    return out


# ---- 1. kernels against the oracle at the maxima ---------------------------------------------------------------------

SIZES = [(1080, 1920), (540, 960), (720, 1280), (480, 640), (641, 1283), (600, 800), (300, 500), (1000, 700)]


def _random_region(rng, h, w, n_poly=8, n_vert=32):
    polys = []
    for p in range(n_poly):
        cx, cy = rng.integers(-w // 4, w + w // 4), rng.integers(-h // 4, h + h // 4)
        rx, ry = rng.integers(8, w // 2 + 9), rng.integers(8, h // 2 + 9)
        polys.append([(int(cx + rng.integers(-rx, rx + 1)), int(cy + rng.integers(-ry, ry + 1))) for _ in range(n_vert)])
    kinds = rng.integers(0, 2, n_poly)
    return ([q for q, k in zip(polys, kinds) if k == 0], [q for q, k in zip(polys, kinds) if k == 1])


def _dets_on(rng, region, h, w, K):
    """K boxes whose anchors lie on the region's vertices, on its edges, on grid ties and anywhere."""
    polys = region[0] + region[1]
    boxes = np.zeros((K, 4), np.float32)
    for k in range(K):
        kind = k % 4
        if kind < 2 and polys:
            q = polys[rng.integers(len(polys))]
            v = rng.integers(len(q))
            a, b = q[v], q[(v + 1) % len(q)]
            px, py = (2 * a[0], 2 * a[1]) if kind == 0 else (a[0] + b[0], a[1] + b[1])  # vertex / edge midpoint
        else:
            px, py = int(rng.integers(-40, 2 * w + 40)), int(rng.integers(-40, 2 * h + 40))
        hw, bh = rng.integers(2, 80) / 2, rng.integers(4, 160) / 2
        x1, x2, y2 = np.float32(px / 2 - hw), np.float32(px / 2 + hw), np.float32(py / 2)
        if kind == 2:  # ties: sums that land on, or round across, an integer; 2 * y2 just below one
            x1 = np.float32(x1 + rng.choice([0.25, 0.5, -0.5, 0.75]))
            if rng.integers(2):
                x1 = np.nextafter(x1, np.float32(-1e9) if rng.integers(2) else np.float32(1e9))
            if rng.integers(2):
                y2 = np.nextafter(y2, np.float32(-1e9))
        elif kind == 3:
            x1, x2 = np.float32(x1 + rng.random()), np.float32(x2 + rng.random())
            y2 = np.float32(y2 + rng.random())
        boxes[k] = (x1, np.float32(y2 - bh), x2, y2)
    return boxes


def _oracle_k5(entries, sizes, dets, filters, regions, min_conf=0.3):
    """K5 outputs as the device defines them: filter (confidence, class), region, crop rectangle, rows in table order."""
    from ai_camera_b200 import config
    boxes, scores, labels, num = (d.cpu().numpy() for d in dets)
    K = scores.shape[1]
    out = dict(det_count=[], det_index=[], crop_slot=[], crop_rect=[])
    for b, e in enumerate(entries):
        if e is None:
            out["det_count"].append(0), out["det_index"].append([]), out["crop_slot"].append([])
            continue
        f = filters[b] if b < len(filters) else None
        mc = np.float32(f.min_confidence if f else min_conf)
        lo, hi = (f.class_mask_lo, f.class_mask_hi) if f else config.tracked_class_mask()
        h, w = sizes[b]
        n = min(int(num[b]), K)
        kept = [i for i in range(n) if scores[b, i] >= mc and 0 <= labels[b, i] < 128 and
                ((lo >> int(labels[b, i])) if labels[b, i] < 64 else (hi >> (int(labels[b, i]) - 64))) & 1 and
                R.keep(regions[b], boxes[b, i])]
        slots = []
        for i in kept:
            x1, y1, x2, y2 = boxes[b, i]
            rect = [max(0, int(x1)), max(0, int(y1)), min(w, int(x2)), min(h, int(y2))]
            if rect[0] < rect[2] and rect[1] < rect[3]:
                slots.append(len(out["crop_rect"]))
                out["crop_rect"].append([b] + rect)
            else:
                slots.append(-1)
        out["det_count"].append(len(kept)), out["det_index"].append(kept), out["crop_slot"].append(slots)
    return out


def test_kernels_equal_the_oracle_at_the_maxima():
    rng = np.random.default_rng(11)
    S, K = 64, 100
    images = {hw: torch.from_numpy(synth_image(rng, *hw)).to(DEV) for hw in SIZES}
    from ai_camera_b200 import synth
    sizes = [SIZES[b % len(SIZES)] for b in range(S)]
    entries = [synth.bgr_to_nv12(images[hw][None])[0].contiguous() if b % 9 == 2 and hw[0] % 2 == hw[1] % 2 == 0
               else images[hw] for b, hw in enumerate(sizes)]
    for b in (5, 17, 40, 63):
        entries[b] = None
    regions = [_random_region(rng, h, w) for h, w in sizes]
    for b in (3, 10, 33, 50):
        regions[b] = ([], [])  # no region
    regions[20] = ([], regions[20][1] + regions[20][0])  # excludes only: the whole frame minus them
    classes = [None, {"person", "car"}, {"bicycle", "truck"}]
    filters = [_filter(float(rng.choice([0.2, 0.3, 0.5])), classes[rng.integers(3)]) for _ in range(40)]  # entries 40.. use the arguments of the call
    boxes = np.stack([_dets_on(rng, regions[b], *sizes[b], K) for b in range(S)])
    scores = rng.choice(np.float32([0.2, 0.35, 0.5, 0.9]), (S, K)).astype(np.float32)
    labels = rng.choice(np.int32([0, 2, 1, 7, 5]), (S, K)).astype(np.int32)
    num = rng.integers(60, K + 1, S).astype(np.int32)
    num[::7] = K
    dets = [torch.from_numpy(a).to(DEV) for a in (boxes, scores, labels, num)]
    cap = S * K
    t = Table(entries, filters)
    try:
        recs = [_record(r) for r in regions]
        _check(_set_regions(t.handle, list(range(S)), recs))
        got = _k5(t, dets, K, cap)
    finally:
        t.close()
    want = _oracle_k5(entries, sizes, dets, filters, regions)
    n_crops = len(want["crop_rect"])
    assert got["crop_count"].tolist() == [n_crops, n_crops]
    assert got["crop_rect"][:n_crops].tolist() == want["crop_rect"]
    dropped = 0
    for b in range(S):
        nb = want["det_count"][b]
        assert int(got["det_count"][b]) == nb, b
        assert got["det_index"][b, :nb].tolist() == want["det_index"][b], b
        assert got["crop_slot"][b, :nb].tolist() == want["crop_slot"][b], b
        if entries[b] is not None and regions[b][0] + regions[b][1]:
            dropped += int(num[b]) - int(R.keep_mask(regions[b], boxes[b, :num[b]]).sum())
    assert dropped > 0 and n_crops > 0
    # the same detections compacted on the host, through a region-less table: the same rows and the same crops
    kept_idx, cb, cs, cl, cn = [], boxes.copy(), scores.copy(), labels.copy(), num.copy()
    for b in range(S):
        m = np.nonzero(R.keep_mask(regions[b], boxes[b, :num[b]]))[0]
        kept_idx.append(m)
        cn[b], cb[b], cs[b], cl[b] = R.compact(regions[b], num[b], boxes[b], scores[b], labels[b])
    t = Table(entries, filters)
    try:
        ref = _k5(t, [torch.from_numpy(a).to(DEV) for a in (cb, cs, cl, cn)], K, cap)
    finally:
        t.close()
    assert torch.equal(got["det_count"], ref["det_count"])
    assert torch.equal(got["crop_count"], ref["crop_count"])
    assert torch.equal(got["crop_rect"][:n_crops], ref["crop_rect"][:n_crops])
    assert torch.equal(got["crops"][:n_crops], ref["crops"][:n_crops])
    for b in range(S):
        nb = int(ref["det_count"][b])
        assert torch.equal(got["crop_slot"][b, :nb], ref["crop_slot"][b, :nb]), b
        assert got["det_index"][b, :nb].tolist() == kept_idx[b][ref["det_index"][b, :nb].numpy()].tolist(), b


# ---- pipelines ------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def blobs(tmp_path_factory):
    from ai_camera_b200 import synth
    return synth.make_blobs(str(tmp_path_factory.mktemp("blobs")))


@pytest.fixture(scope="module")
def bias(blobs):
    from ai_camera_b200 import synth
    return synth.shifted_class_bias(blobs[0], -0.6)


def _pipeline(blobs, bias, n, settings=None, **kw):
    from ai_camera_b200 import synth
    from ai_camera_b200.pipeline import TrackingPipeline
    p = TrackingPipeline(blobs[0], blobs[1], n, max_tracks=128, stream_settings=settings, **kw)
    synth.apply_class_bias(p.detector.engine, bias)
    return p


def _video(h, w, seed, n_frames):
    from ai_camera_b200 import synth
    return synth.SynthVideo(1, (h, w), n_frames=n_frames, seed=seed).ring[:, 0]


def _rows(ot, oc, on, s):
    from ai_camera_b200 import config
    return [tuple(int(v) for v in ot[s, k, :5]) + (config.CLASSES[ot[s, k, 5]], float(oc[s, k])) for k in range(on[s])]


def _box(x0, y0, x1, y1):
    return ((x0, y0), (x1, y0), (x1, y1), (x0, y1))


U = ((0, 0), (960, 0), (960, 540), (640, 540), (640, 180), (320, 180), (320, 540), (0, 540))


def _region_settings():
    from ai_camera_b200.pipeline import StreamSettings
    return [StreamSettings(n_init=2, include_regions=[_box(0, 0, 480, 540)]),                   # left half
            StreamSettings(n_init=2, exclude_regions=[_box(0, 0, 1280, 300)]),                  # top strip
            StreamSettings(n_init=2),                                                            # none
            StreamSettings(n_init=1, include_regions=[U], exclude_regions=[_box(0, 0, 200, 200)]),
            StreamSettings(n_init=2, include_regions=[_box(0, 0, 600, 600), _box(300, 200, 960, 540)],
                           exclude_regions=[_box(400, 250, 520, 400)])]


SIZES_P = [(540, 960), (720, 1280), (540, 960), (540, 960), (540, 960)]


def _without_regions(st):
    return replace(st, include_regions=(), exclude_regions=())


def test_tracking_equals_a_regionless_tracker_on_compacted_detections(blobs, bias):
    from ai_camera_b200.pipeline import BatchTracker
    settings = _region_settings()
    S, T = len(settings), 32
    videos = [_video(h, w, 300 + s, 16) for s, (h, w) in enumerate(SIZES_P)]
    pipe = _pipeline(blobs, bias, S, settings)
    ref = BatchTracker(blobs[1], S, max_dets=pipe.detector.topk, max_tracks=128,
                       min_detection_confidence=pipe.tracker.min_conf)
    ref.configure_streams(range(S), [_without_regions(st) for st in settings])
    oracle_regions = [(list(st.include_regions), list(st.exclude_regions)) for st in settings]
    dropped, kept, reported = [0] * S, [0] * S, [0] * S
    for t in range(T):
        k = t % 30 if t % 30 < 16 else 30 - t % 30
        frames = [None if (s == 3 and t in (7, 19)) else videos[s][k] for s in range(S)]
        got = [x.cpu().numpy() for x in pipe.step(frames)]
        num, boxes, scores, labels = (x.cpu().numpy().copy() for x in (pipe.detector.num_dets, pipe.detector.boxes,
                                                                      pipe.detector.scores, pipe.detector.labels))
        for s in range(S):
            n0 = int(num[s])
            num[s], boxes[s], scores[s], labels[s] = R.compact(oracle_regions[s], num[s], boxes[s], scores[s], labels[s])
            dropped[s] += n0 - int(num[s])
            kept[s] += int(num[s])
        want = [x.cpu().numpy() for x in ref.update(frames, *[torch.from_numpy(a).to(DEV) for a in (num, boxes, scores,
                                                                                                   labels)])]
        assert np.array_equal(got[2], want[2]), t
        for s in range(S):
            assert _rows(*got, s) == _rows(*want, s), (t, s)
            a, b = pipe.tracker.snapshot(s), ref.snapshot(s)
            assert np.array_equal(a[0], b[0]) and np.array_equal(a[1].view(np.uint32), b[1].view(np.uint32)), (t, s)
            reported[s] += int(got[2][s])
    for s, st in enumerate(settings):
        assert reported[s] > 0, (s, reported)
        if st.has_regions():
            assert dropped[s] > 0 and kept[s] > 0, (s, dropped, kept)
    assert not pipe.tracker.overflow().any()


def _pass_all():
    from ai_camera_b200.pipeline import StreamSettings
    edge = [(-LIMIT + k * (2 * LIMIT // 8), -LIMIT) for k in range(8)] + [(LIMIT, -LIMIT + k * (2 * LIMIT // 8))
                                                                          for k in range(8)]
    edge += [(LIMIT - k * (2 * LIMIT // 8), LIMIT) for k in range(8)] + [(-LIMIT, LIMIT - k * (2 * LIMIT // 8))
                                                                        for k in range(8)]
    off = [[(-5000 - 10 * k - j, -100 - (j * j) % 50) for j in range(32)] for k in range(7)]  # left of every frame
    return StreamSettings(n_init=2, include_regions=[edge], exclude_regions=off)


def test_pass_all_region_changes_nothing_but_one_launch(blobs, bias):
    from ai_camera_b200 import synth
    from ai_camera_b200.pipeline import StreamSettings
    S = 4
    video = synth.SynthVideo(S, (540, 960), n_frames=5, seed=31)
    plain = _pipeline(blobs, bias, S, n_init=2)
    neutral = _pipeline(blobs, bias, S, [StreamSettings(n_init=2)] * S, n_init=2)
    passall = _pipeline(blobs, bias, S, [_pass_all()] * S, n_init=2)
    assert passall.settings[0].resolve_region().n_polygons == 8
    lib = _lib()
    pipes = (plain, neutral, passall)
    for p in pipes:  # (warm: first sights of sizes and paths)
        p.step(list(video.frames(0)))
        p.step(video.frames(0))
        p.tracker.reset()
    torch.cuda.synchronize()
    total = 0
    for as_list in (True, False):
        for t in range(5):
            frames = list(video.frames(t)) if as_list else video.frames(t)
            outs, counts = [], []
            for p in pipes:
                before = lib.aicam_launch_count()
                outs.append([x.cpu().clone() for x in p.step(frames)])
                counts.append(lib.aicam_launch_count() - before)
            for o in outs[1:]:
                assert all(torch.equal(a, b) for a, b in zip(outs[0], o)), (as_list, t)
            if as_list:
                list_count = counts[0]
            # (a stacked step with regions runs as a list step: one more launch than the list step without them)
            assert counts[0] == counts[1] and counts[2] == list_count + 1, counts
            assert passall.launches_per_step(as_list) == plain.launches_per_step(True) + 1
            total += int(outs[0][2].sum())
        for p in pipes:
            p.tracker.reset()
    assert total > 0
    # a pipeline that never sets a region makes the launches it made before regions existed
    assert neutral.launches_per_step() == plain.launches_per_step()
    tr = plain.tracker
    assert tr.launches_per_step() == 5 + tr.reid.launches_per_forward() - (1 if tr._nhwc8 else 0)


def test_stacked_step_equals_the_list_step(blobs, bias):
    from ai_camera_b200 import synth
    settings = [st for st, hw in zip(_region_settings(), SIZES_P) if hw == (540, 960)]
    S = len(settings)
    video = synth.SynthVideo(S, (540, 960), n_frames=6, seed=41)
    stacked, listed = _pipeline(blobs, bias, S, settings), _pipeline(blobs, bias, S, settings)
    total = 0
    for t in range(6):
        a = [x.cpu().numpy() for x in stacked.step(video.frames(t))]
        b = [x.cpu().numpy() for x in listed.step(list(video.frames(t)))]
        assert np.array_equal(a[2], b[2]), t
        for s in range(S):
            assert _rows(*a, s) == _rows(*b, s), (t, s)
        total += int(a[2].sum())
    assert total > 0
    assert stacked.launches_per_step() == stacked.launches_per_step(True)


def test_captured_step_follows_region_and_presence_changes(blobs, bias):
    from ai_camera_b200.pipeline import StreamSettings
    sizes = [(540, 960), (1080, 1920), (480, 640)]
    T = 7
    videos = [_video(h, w, 330 + i, T) for i, (h, w) in enumerate(sizes)]
    masks = [[1, 1, 1], [1, 0, 1], [1, 1, 1], [0, 1, 1], [1, 1, 0], [1, 1, 1], [1, 1, 1]]
    first = [StreamSettings(n_init=1, include_regions=[_box(0, 0, 480, 540)]), StreamSettings(n_init=1),
             StreamSettings(n_init=1, exclude_regions=[_box(0, 240, 640, 480)])]
    changes = {1: ([1], [StreamSettings(n_init=1, exclude_regions=[_box(0, 0, 1920, 500), U])]),
               3: ([0, 2], [StreamSettings(n_init=1), StreamSettings(n_init=1, include_regions=[_box(100, 0, 400, 480)])]),
               5: ([0, 1, 2], [StreamSettings(n_init=1)] * 3)}  # every region cleared
    g_pipe, e_pipe = (_pipeline(blobs, bias, 3, first, max_frame_hw=(1080, 1920)) for _ in range(2))
    g_pipe.step([v[0] for v in videos])
    torch.cuda.synchronize()
    g_pipe.tracker.reset()
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=stream):
        out = g_pipe.step_table()
    reported = 0
    for t in range(T):
        if t in changes:
            for p in (g_pipe, e_pipe):
                p.configure_streams(*changes[t])
        frames = [videos[s][t] if masks[t][s] else None for s in range(3)]
        g_pipe.frame_table.set(frames)
        g.replay()
        want = e_pipe.step(frames)
        torch.cuda.synchronize()
        got = [x.cpu().numpy() for x in out]
        want = [x.cpu().numpy() for x in want]
        assert np.array_equal(got[2], want[2]), t
        for s in range(3):
            assert _rows(*got, s) == _rows(*want, s), (t, s)
        reported += int(want[2].sum())
    assert reported > 0


def test_resets_keep_or_take_regions(blobs, bias):
    from ai_camera_b200.pipeline import StreamSettings
    left = StreamSettings(n_init=1, include_regions=[_box(0, 0, 480, 540)])
    lower = StreamSettings(n_init=1, exclude_regions=[_box(0, 0, 960, 270)])
    T, Rs = 8, 4
    videos = [_video(540, 960, 360 + i, T) for i in range(2)]
    new_src = [_video(540, 960, 370 + i, T - Rs) for i in range(2)]
    pipe = _pipeline(blobs, bias, 2, [left, lower])
    fresh = [_pipeline(blobs, bias, 1, [st]) for st in (left, lower, left, left)]
    total = 0
    for t in range(T):
        if t == Rs:
            pipe.reset_streams([0])                 # keeps `left`
            pipe.reset_streams([1], settings=left)  # takes `left`
        frames = [v[t] for v in videos] if t < Rs else [new_src[0][t - Rs], new_src[1][t - Rs]]
        got = [x.cpu().numpy() for x in pipe.step(frames)]
        for s in range(2):
            ref = fresh[s] if t < Rs else fresh[2 + s]
            want = _rows(*[x.cpu().numpy() for x in ref.step([frames[s]])], 0)
            assert _rows(*got, s) == want, (t, s)
            total += len(want)
    assert pipe.settings == [left, left] and total > 0


# ---- 5. ABI validation ----------------------------------------------------------------------------------------------

def test_abi_rejects_bad_regions_and_changes_nothing():
    L = _L()
    rng = np.random.default_rng(3)
    sizes = [(540, 960), (480, 640), (720, 1280)]
    frames = [torch.from_numpy(synth_image(rng, h, w)).to(DEV) for h, w in sizes]
    K = 40
    region = ([[(0, 0), (300, 0), (300, 500), (0, 500)]], [[(50, 50), (120, 50), (120, 300)]])
    boxes = np.stack([_dets_on(rng, region, h, w, K) for h, w in sizes])
    dets = [torch.from_numpy(a).to(DEV) for a in (boxes, np.full((3, K), 0.9, np.float32), np.zeros((3, K), np.int32),
                                                   np.full(3, K, np.int32))]
    lib = _lib()
    t, fresh = Table(frames), Table(frames)
    try:
        before_any = lib.aicam_launch_count()
        _k5(fresh, dets, K, 3 * K)
        plain_launches = lib.aicam_launch_count() - before_any

        def bad(**kw):
            r = _record(region)
            for k, v in kw.items():
                if k == "xy":
                    r.xy[0][1][v[0]] = v[1]
                elif k in ("kind", "n_vertices"):
                    getattr(r, k)[0] = v
                else:
                    setattr(r, k, v)
            return r
        cases = [([3], [_record(region)]), ([-1], [_record(region)]), ([0], [bad(n_polygons=9)]),
                 ([0], [bad(n_polygons=-1)]), ([0], [bad(kind=2)]), ([0], [bad(kind=-1)]), ([0], [bad(n_vertices=2)]),
                 ([0], [bad(n_vertices=33)]), ([0], [bad(xy=(0, LIMIT + 1))]), ([0], [bad(xy=(1, -LIMIT - 1))]),
                 ([0, 1], [_record(region), bad(kind=5)])]  # (the valid first entry is not stored either)
        before = lib.aicam_launch_count()
        for idx, recs in cases:
            assert _set_regions(fresh.handle, idx, recs) == -1, (idx, recs)
        assert lib.aicam_frame_table_set_regions(fresh.handle, None, None, 1, None) == -1
        assert lib.aicam_frame_table_set_regions(fresh.handle, (C.c_int32 * 1)(0), None, -1, None) == -1
        assert lib.aicam_launch_count() == before
        # a table whose every region call was rejected has no region test
        before = lib.aicam_launch_count()
        after_bad = _k5(fresh, dets, K, 3 * K)
        assert lib.aicam_launch_count() - before == plain_launches
        ref = _k5(t, dets, K, 3 * K)
        assert all(torch.equal(after_bad[k], ref[k]) for k in ref)
        # with a region: the step after rejected calls equals the one before them
        _check(_set_regions(t.handle, [1], [_record(region)]))
        one = _k5(t, dets, K, 3 * K)
        for idx, recs in cases:
            assert _set_regions(t.handle, idx, recs) == -1
        two = _k5(t, dets, K, 3 * K)
        assert all(torch.equal(one[k], two[k]) for k in one)
        assert int(one["det_count"][1]) < K and int(one["det_count"][0]) == K
        # an empty record clears the entry; the test keeps launching
        _check(_set_regions(t.handle, [1], [L.StreamRegion()]))
        before = lib.aicam_launch_count()
        cleared = _k5(t, dets, K, 3 * K)
        assert lib.aicam_launch_count() - before == plain_launches + 1
        assert all(torch.equal(cleared[k], ref[k]) for k in ref)
        # the region test takes at most 1024 detections per frame
        big = [torch.zeros((3, 1025, 4), device=DEV), torch.zeros((3, 1025), device=DEV),
               torch.zeros((3, 1025), dtype=torch.int32, device=DEV), torch.zeros(3, dtype=torch.int32, device=DEV)]
        with pytest.raises(L.AicamError) as e:
            _k5(t, big, 1025, 8)
        assert e.value.code == -4
    finally:
        t.close()
        fresh.close()


# ---- 6. command line ------------------------------------------------------------------------------------------------

def _write_clip(path, frames):
    import cv2
    w = cv2.VideoWriter(str(path), cv2.VideoWriter_fourcc(*"mp4v"), 10, (frames[0].shape[1], frames[0].shape[0]))
    for f in frames:
        w.write(f)
    w.release()
    return str(path)


def test_cli_runs_each_input_with_its_regions(blobs, tmp_path):
    import cv2
    from ai_camera_b200 import synth, weights
    from ai_camera_b200.aicamera_tracker import main, run_batched, tracks_to_rows, video_frames
    from ai_camera_b200.pipeline import StreamSettings, TrackingPipeline
    kind, params, tensors = weights.read_blob(blobs[0])
    tensors = dict(tensors)
    for n, b in synth.shifted_class_bias(blobs[0], synth.CLIP_LOGIT_SHIFT).items():
        tensors[n + ".bias"] = b
    yolo = weights.write_blob(str(tmp_path / "yolo_clip.aicw"), kind, params, tensors)
    clip = list(video_frames(CLIP, 10))
    h, w = clip[0].shape[:2]
    paths = [_write_clip(tmp_path / "a.mp4", clip), _write_clip(tmp_path / "b.mp4", [cv2.resize(f, (1280, 720)) for f in clip])]
    spec = {"default": {"n_init": 2},
            "a.mp4": {"exclude_regions": [[[0, 0], [w, 0], [w, h // 2], [0, h // 2]]]},
            "b.mp4": {"include_regions": [[[0, 0], [850, 0], [850, 720], [0, 720]], [[900, 400], [1280, 400], [1280, 720]]],
                      "exclude_regions": [[[100, 100], [300, 100], [300, 300], [100, 300]]]}}
    (tmp_path / "s.json").write_text(json.dumps(spec))
    out = tmp_path / "out"
    argv = sum((["--input", p] for p in paths), []) + ["--streams", "2", "--stream_settings", str(tmp_path / "s.json"),
                                                     "--output_dir", str(out), "--output_filename", "run",
                                                     "--yolo_engine", yolo, "--reid_engine", blobs[1]]
    assert main(argv) == 0
    lines = [json.loads(l) for l in open(out / "run.tracks.jsonl")]
    total = 0
    for s, p in enumerate(paths):
        st = StreamSettings.from_dict(spec[os.path.basename(p)], StreamSettings.from_dict(spec["default"]))
        assert st.has_regions()
        one = TrackingPipeline(yolo, blobs[1], 1, stream_settings=[st])
        want = []
        run_batched([video_frames(p)], one, lambda step, batch, table: want.append(tracks_to_rows([x.numpy() for x in table], 0)))
        got = [[tuple(r) for r in l["tracks"]] for l in sorted((l for l in lines if l["stream"] == s), key=lambda l: l["frame"])]
        assert got == want, p
        total += sum(len(r) for r in want)
    assert total > 0
