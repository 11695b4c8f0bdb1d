"""Per-stream detection and tracking settings in one batched step: per-entry NMS thresholds, confidence and class mask in
the frame table (aicam_frame_table_set_filters), per-stream association settings in the tracker
(aicam_tracker_set_stream_assoc), StreamSettings / configure_streams / reset_streams(settings=) on the pipeline, and the
--stream_settings flag.  The GPU tests (-m gpu) compare bit for bit against the same work run alone with those settings;
the tests without the mark check the host side."""
import ctypes as C
import json
import os

import numpy as np
import pytest
import torch

from scenarios import make_scenario, synth_image

DEV = torch.device("cuda:0")
CLIP = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "aicamera_test_clip.mp4")
gpu = pytest.mark.gpu


def _L():
    from ai_camera_b200 import _lib as L
    return L


def _lib():
    return _L().load()


def _check(rc):
    _L().check(rc)


# ---- host side ------------------------------------------------------------------------------------------------------

def test_resolver_follows_the_constructor_rule():
    from ai_camera_b200 import config
    from ai_camera_b200.pipeline import StreamSettings, resolve_thresholds
    assert resolve_thresholds(0.5) == (config.YOLO_CONF_THRESHOLD, 0.5)
    assert resolve_thresholds(0.2) == (0.2, config.DEEPSORT_MIN_CONFIDENCE)
    assert resolve_thresholds(0.2, 0.1) == (0.2, 0.1)
    f, a = StreamSettings(conf_threshold=0.5, nms_threshold=0.4, classes_to_track={"car", "truck"}, max_age=10,
                          n_init=1, max_cosine_distance=0.25).resolve()
    assert (f.score_thr, f.iou_thr, f.min_confidence) == (np.float32(0.3), np.float32(0.4), np.float32(0.5))
    assert (f.class_mask_lo, f.class_mask_hi) == ((1 << 2) | (1 << 7), 0)
    assert (a.max_cosine_distance, a.max_iou_distance, a.max_age, a.n_init) == (0.25, config.DEEPSORT_MAX_IOU_DISTANCE, 10, 1)
    f, a = StreamSettings().resolve()
    assert (f.class_mask_lo, f.class_mask_hi) == config.tracked_class_mask()
    assert (a.max_age, a.n_init) == (config.DEEPSORT_MAX_AGE, config.DEEPSORT_N_INIT)


@pytest.mark.parametrize("kw", [dict(conf_threshold=float("nan")), dict(conf_threshold=1.5), dict(nms_threshold=-0.1),
                                dict(min_detection_confidence=2.0), dict(max_age=0), dict(max_age=256), dict(n_init=0),
                                dict(max_cosine_distance=float("inf")), dict(max_iou_distance=-1.0),
                                dict(classes_to_track={"car", "unicorn"}), dict(classes_to_track="car")])
def test_stream_settings_reject_bad_values(kw):
    from ai_camera_b200.pipeline import StreamSettings
    with pytest.raises(ValueError):
        StreamSettings(**kw)


def test_stream_settings_file(tmp_path):
    from ai_camera_b200.aicamera_tracker import load_stream_settings, parse_arguments
    from ai_camera_b200.pipeline import StreamSettings
    p = tmp_path / "s.json"
    p.write_text(json.dumps({"default": {"max_age": 30}, "a.mp4": {"classes_to_track": ["car", "truck"],
                                                                     "conf_threshold": 0.5}}))
    get = load_stream_settings(str(p), 0.25)
    assert get("a.mp4") == StreamSettings(conf_threshold=0.5, classes_to_track={"car", "truck"}, max_age=30)
    assert get("b.mp4") == get(None) == StreamSettings(conf_threshold=0.25, max_age=30)
    args = parse_arguments(["--input", "x/a.mp4", "--streams", "2", "--stream_settings", str(p)])
    assert args.settings_for("a.mp4").classes_to_track == {"car", "truck"}
    assert parse_arguments(["--input", "a.mp4"]).settings_for is None
    for bad in ({"a.mp4": {"max_agee": 3}}, {"a.mp4": {"n_init": 0}}, ["not", "an", "object"]):
        p.write_text(json.dumps(bad))
        with pytest.raises(SystemExit):
            parse_arguments(["--input", "a.mp4", "--streams", "1", "--stream_settings", str(p)])
    with pytest.raises(SystemExit):  # single-stream mode takes the facades' arguments
        parse_arguments(["--input", "a.mp4", "--stream_settings", str(p)])


# ---- device: frame table and kernels --------------------------------------------------------------------------------

def _filter(score=0.3, iou=0.5, min_conf=0.3, classes=None):
    from ai_camera_b200 import config
    lo, hi = config.tracked_class_mask(classes)
    return _L().StreamFilter(score, iou, min_conf, 0, lo, hi)


class Table:
    """A frame table with per-entry filters (None: none), set from entries (None = absent): BGR [H, W, 3] / NV12
    [H*3/2, W] tensors."""

    def __init__(self, entries, filters=None):
        L = _L()
        self.handle = C.c_void_p()
        _check(_lib().aicam_frame_table_create(0, len(entries), 2160, 3840, C.byref(self.handle)))
        if filters:
            _check(_lib().aicam_frame_table_set_filters(self.handle, (L.StreamFilter * len(filters))(*filters), len(filters)))
        descs = (L.FrameDesc * len(entries))()
        for d, e in zip(descs, entries):
            if e is None:
                continue
            if e.dim() == 3:
                d.data, d.chroma, d.h, d.w, d.pitch, d.kind = e.data_ptr(), None, e.shape[0], e.shape[1], e.stride(0), 0
            else:
                h = e.shape[0] * 2 // 3
                d.data, d.chroma, d.h, d.w, d.pitch, d.kind = (e.data_ptr(), e.data_ptr() + h * e.stride(0), h, e.shape[1],
                                                               e.stride(0), 1)
        present = (C.c_uint8 * len(entries))(*[e is not None for e in entries])
        _check(_lib().aicam_frame_table_set_present(self.handle, descs, present, len(entries), None))
        self.n = len(entries)

    def close(self):
        _lib().aicam_frame_table_destroy(self.handle)


def _nv12(frame_bgr):
    from ai_camera_b200 import synth
    return synth.bgr_to_nv12(frame_bgr[None])[0].contiguous()


def _video(h, w, seed, n_frames=1):
    from ai_camera_b200 import synth
    return synth.SynthVideo(1, (h, w), n_frames=n_frames, seed=seed).ring[:, 0]


@pytest.fixture(scope="module")
def blobs(tmp_path_factory):
    from ai_camera_b200 import synth
    return synth.make_blobs(str(tmp_path_factory.mktemp("blobs")))


@pytest.fixture(scope="module")
def bias(blobs):
    from ai_camera_b200 import synth
    return synth.shifted_class_bias(blobs[0], -0.6)


@gpu
def test_detect_with_per_entry_settings(blobs, bias):
    from ai_camera_b200 import synth
    from ai_camera_b200.pipeline import BatchDetector
    sizes = [(1080, 1920), (540, 960), (720, 1280), (480, 640), (641, 1283), (1080, 1920), (600, 800)]
    frames = [_video(h, w, 40 + i)[0] for i, (h, w) in enumerate(sizes)]
    frames[2] = _nv12(frames[2])
    entries = list(frames)
    entries[3] = None
    # entries 0-4 carry settings (entry 4 the entry points' own values), 5 and 6 use the entry points' arguments
    settings = [(0.45, 0.3), (0.2, 0.7), (0.3, 0.4), (0.6, 0.2), (0.3, 0.5)]
    det = BatchDetector(blobs[0], len(frames))
    synth.apply_class_bias(det.engine, bias)

    def run(table):
        out = det.detect_table(table)
        torch.cuda.synchronize()
        return [o.cpu().clone() for o in out]

    def alone(frame, score, iou):
        det._nms.score_thr, det._nms.iou_thr = score, iou
        try:
            out = det.detect(frame[None])
            torch.cuda.synchronize()
            return [o.cpu().clone() for o in out]
        finally:
            det._nms.score_thr, det._nms.iou_thr = det.engine.score_threshold, det.engine.nms_threshold
    t = Table(entries, [_filter(s, i) for s, i in settings])
    try:
        got = run(t)
    finally:
        t.close()
    seen, differs = 0, False
    for b, e in enumerate(entries):
        if e is None:
            assert int(got[0][b]) == 0 and not any(bool(g[b].any()) for g in got[1:])
            continue
        score, iou = settings[b] if b < len(settings) else (det.engine.score_threshold, det.engine.nms_threshold)
        want = alone(e, score, iou)
        for g, w in zip(got, want):
            assert torch.equal(g[b], w[0]), b
        seen += int(want[0][0])
        if b < 4:  # (the settings change what is detected)
            differs |= not all(torch.equal(g[b], w[0]) for g, w in zip(got, alone(e, 0.3, 0.5)))
    assert seen > 0 and differs
    # an all-absent table with settings stays empty
    t = Table([None] * len(frames), [_filter(0.1, 0.9)] * len(frames))
    try:
        assert not any(bool(g.any()) for g in run(t))
    finally:
        t.close()


def _dets_for(sizes, rng, K=24):
    n = len(sizes)
    boxes = np.zeros((n, K, 4), np.float32)
    for b, (h, w) in enumerate(sizes):
        for k in range(K):
            x, y = rng.uniform(-20, w), rng.uniform(-20, h)
            boxes[b, k] = (x, y, x + rng.uniform(2, 0.4 * w + 3), y + rng.uniform(2, 0.6 * h + 3))
    scores = rng.choice(np.float32([0.2, 0.35, 0.5, 0.9]), (n, K)).astype(np.float32)
    labels = rng.choice(np.int32([0, 2, 1, 7, 5]), (n, K)).astype(np.int32)
    num = rng.integers(K // 2, K + 1, n).astype(np.int32)
    return [torch.from_numpy(a).to(DEV) for a in (boxes, scores, labels, num)]


def _k5(target, dets, min_conf, mask):
    boxes, scores, labels, num = dets
    B, K = scores.shape
    cap = B * K
    i32 = dict(dtype=torch.int32, device=DEV)
    o = dict(det_index=torch.full((B, K), -7, **i32), det_count=torch.full((B,), -7, **i32),
             crop_slot=torch.full((B, K), -7, **i32), crop_rect=torch.zeros((cap, 5), **i32),
             crops=torch.zeros((cap, 128, 64, 8), dtype=torch.bfloat16, device=DEV), crop_count=torch.zeros(2, **i32))
    tail = (boxes.data_ptr(), scores.data_ptr(), labels.data_ptr(), num.data_ptr(), K, min_conf, mask[0], mask[1], 2, cap,
            o["det_index"].data_ptr(), o["det_count"].data_ptr(), o["crop_slot"].data_ptr(), o["crop_rect"].data_ptr(),
            o["crops"].data_ptr(), o["crop_count"].data_ptr(), None)
    if isinstance(target, Table):
        _check(_lib().aicam_reid_crops_table(target.handle, *tail))
    elif target.dim() == 3:
        _check(_lib().aicam_reid_crops(target.data_ptr(), 1, target.shape[0], target.shape[1], *tail))
    else:
        _check(_lib().aicam_reid_crops_nv12(target.data_ptr(), 1, target.shape[0] * 2 // 3, target.shape[1], *tail))
    torch.cuda.synchronize()
    out = {k: v.cpu() for k, v in o.items()}
    out["n"] = int(out["crop_count"][0])
    return out


@gpu
def test_crop_filter_with_per_entry_settings():
    from ai_camera_b200 import config
    rng = np.random.default_rng(5)
    sizes = [(540, 960), (480, 640), (1080, 1920), (101, 37), (720, 1280)]
    frames = [torch.from_numpy(synth_image(rng, h, w)).to(DEV) for h, w in sizes]
    frames[1] = _nv12(frames[1])
    dets = _dets_for(sizes, rng)
    settings = [(0.5, {"car", "truck"}), (0.2, {"person"}), (0.9, None), (0.35, {"bicycle", "person", "bus"})]
    t = Table(frames, [_filter(min_conf=m, classes=c) for m, c in settings])  # entry 4: the arguments below
    try:
        got = _k5(t, dets, 0.3, config.tracked_class_mask())
    finally:
        t.close()
    base = 0
    for b, f in enumerate(frames):
        m, c = settings[b] if b < len(settings) else (0.3, None)
        one = _k5(f, [d[b:b + 1] for d in dets], m, config.tracked_class_mask(c))
        nb = int(one["det_count"][0])
        assert int(got["det_count"][b]) == nb, b
        assert torch.equal(got["det_index"][b, :nb], one["det_index"][0, :nb]), b
        slots = one["crop_slot"][0, :nb]
        assert torch.equal(got["crop_slot"][b, :nb], torch.where(slots >= 0, slots + base, slots)), b
        for k in range(one["n"]):
            assert got["crop_rect"][base + k].tolist() == [b] + one["crop_rect"][k, 1:].tolist()
            assert torch.equal(got["crops"][base + k], one["crops"][k])
        base += one["n"]
    assert got["n"] == base and base > 0
    kept = [int(got["det_count"][b]) for b in range(len(frames))]
    assert kept[1] > 0 and kept[0] > 0


# ---- device: association --------------------------------------------------------------------------------------------

ASSOC = [(0.2, 0.7, 70, 3), (0.3, 0.5, 1, 1), (0.1, 0.9, 255, 2), (0.25, 0.6, 5, 1)]


def _set_assoc(trk_h, indices, values):
    L = _L()
    arr = (L.StreamAssoc * len(values))(*[L.StreamAssoc(*v) for v in values])
    return _lib().aicam_tracker_set_stream_assoc(trk_h, (C.c_int32 * len(indices))(*indices), arr, len(values), None)


def _golden_append(acc, out, snap):
    (o, c), (ints, floats) = out, snap
    acc.setdefault("out", []).extend(o.tolist())
    acc.setdefault("out_conf", []).extend(c.tolist())
    acc.setdefault("out_off", [0]).append(len(acc["out"]))
    acc.setdefault("trk_i", []).extend(ints.tolist())
    acc.setdefault("trk_f", []).extend(floats.tolist())
    acc.setdefault("trk_off", [0]).append(len(acc["trk_i"]))


def _golden(acc):
    return dict(out=np.asarray(acc["out"], np.int64).reshape(-1, 6), out_conf=np.asarray(acc["out_conf"], np.float64),
                out_off=np.asarray(acc["out_off"], np.int64), trk_i=np.asarray(acc["trk_i"], np.int64).reshape(-1, 7),
                trk_f=np.asarray(acc["trk_f"], np.float32).reshape(-1, 25), trk_off=np.asarray(acc["trk_off"], np.int64))


def _oracle_kw(v):
    return dict(max_cosine_distance=v[0], max_iou_distance=v[1], max_age=v[2], n_init=v[3])


@gpu
def test_association_per_stream_equals_the_oracle():
    import gpu_util as G
    from golden_util import assert_same_tracking, run_oracle
    scen = [make_scenario(seed=20 + s, n_frames=40, n_objects=8, feat_dim=64, p_miss=0.2) for s in range(len(ASSOC))]
    kmax = max(len(f["boxes"]) for sc in scen for f in sc)
    trk = G.Tracker(len(ASSOC), max_dets=kmax, feature_dim=64, stride_k=kmax)
    try:
        _check(_set_assoc(trk.h, list(range(len(ASSOC))), ASSOC))
        acc = [{} for _ in ASSOC]
        for t in range(40):
            outs = trk.step([sc[t] for sc in scen])
            for s in range(len(ASSOC)):
                _golden_append(acc[s], outs[s], trk.snapshot(s))
        for s, v in enumerate(ASSOC):
            assert_same_tracking(_golden(acc[s]), run_oracle(scen[s], **_oracle_kw(v)), "stream %d %s" % (s, v))
        assert not trk.overflow().any()
    finally:
        trk.close()


@gpu
def test_settings_change_between_steps_equals_a_changed_reference():
    """Stream 1 changes every association setting at step k, max_age down while its old tracks are live: it equals an
    oracle whose attributes change at the same step (old tracks keep the n_init / max_age they were created with); the
    other streams equal a run without the change."""
    import gpu_util as G
    from golden_util import assert_same_tracking
    from oracle.tracker import DeepSORT
    S, T, k = 3, 40, 15
    old, new = (0.2, 0.7, 70, 3), (0.3, 0.5, 2, 1)
    scen = [make_scenario(seed=50 + s, n_frames=T, n_objects=8, feat_dim=64, p_miss=0.25) for s in range(S)]
    kmax = max(len(f["boxes"]) for sc in scen for f in sc)
    a, b = (G.Tracker(S, max_dets=kmax, feature_dim=64, stride_k=kmax) for _ in range(2))
    oracle = DeepSORT(**_oracle_kw(old))
    acc, want = {}, {}
    try:
        for t in range(T):
            if t == k:
                live = len(b.snapshot(1)[0])
                _check(_set_assoc(b.h, [1], [new]))
                core = oracle.tracker_core
                core.max_cosine_distance, core.max_iou_distance, core.max_age, core.n_init = new
                assert live > 0
            frames = [sc[t] for sc in scen]
            a.step(frames)
            outs = b.step(frames)
            _golden_append(acc, outs[1], b.snapshot(1))
            res = oracle.update(scen[1][t]["boxes"], scen[1][t]["scores"], scen[1][t]["classes"], frame_hw=(1080, 1920),
                                planted_features=scen[1][t]["feats"])
            from oracle.constants import CLASSES
            want.setdefault("out", []).extend([[x1, y1, x2, y2, i, CLASSES.index(c)] for x1, y1, x2, y2, i, c, _ in res])
            want.setdefault("out_conf", []).extend([cf for *_, cf in res])
            want.setdefault("out_off", [0]).append(len(want["out"]))
            tr = oracle.tracker_core.tracks
            want.setdefault("trk_i", []).extend([[x.track_id, x.state, x.hits, x.age, x.time_since_update, x.class_id,
                                                  len(x.features)] for x in tr])
            want.setdefault("trk_f", []).extend([np.concatenate([x.mean, x.cov, [np.float32(x.confidence)]]) for x in tr])
            want.setdefault("trk_off", [0]).append(len(want["trk_i"]))
            for s in (0, 2):
                sa, sb = a.snapshot(s), b.snapshot(s)
                assert np.array_equal(sa[0], sb[0]) and np.array_equal(sa[1].view(np.uint32), sb[1].view(np.uint32)), (t, s)
        assert_same_tracking(_golden(acc), _golden(want), "changed stream")
    finally:
        a.close()
        b.close()


@gpu
def test_validation_rejects_and_changes_nothing(blobs, bias):
    import gpu_util as G
    L, lib = _L(), _lib()
    scen = make_scenario(seed=9, n_frames=12, n_objects=6, feat_dim=64)
    kmax = max(len(f["boxes"]) for f in scen)
    a, b = (G.Tracker(2, max_dets=kmax, feature_dim=64, stride_k=kmax) for _ in range(2))
    try:
        _check(_set_assoc(a.h, [1], [(0.3, 0.5, 5, 1)]))
        _check(_set_assoc(b.h, [1], [(0.3, 0.5, 5, 1)]))
        for t in range(6):
            a.step([scen[t], scen[t]])
            b.step([scen[t], scen[t]])
        bad = [([0], [(0.2, 0.7, 0, 3)]), ([0], [(0.2, 0.7, 256, 3)]), ([0], [(0.2, 0.7, 70, 0)]),
               ([0], [(float("nan"), 0.7, 70, 3)]), ([0], [(0.2, -0.1, 70, 3)]), ([0], [(0.2, float("inf"), 70, 3)]),
               ([2], [(0.2, 0.7, 70, 3)]), ([-1], [(0.2, 0.7, 70, 3)]),
               ([0, 1], [(0.1, 0.9, 9, 2), (0.2, 0.7, 70, 0)])]  # (the valid first entry is not stored either)
        before = lib.aicam_launch_count()
        for idx, vals in bad:
            assert _set_assoc(b.h, idx, vals) == -1, (idx, vals)
        assert lib.aicam_tracker_set_stream_assoc(b.h, None, None, 1, None) == -1
        assert lib.aicam_launch_count() == before
        for t in range(6, 12):
            oa, ob = a.step([scen[t], scen[t]]), b.step([scen[t], scen[t]])
            for s in range(2):
                assert all(np.array_equal(x, y) for x, y in zip(oa[s], ob[s])), (t, s)
                assert np.array_equal(a.snapshot(s)[1].view(np.uint32), b.snapshot(s)[1].view(np.uint32))
    finally:
        a.close()
        b.close()
    # frame-table filters: every bad call stores nothing, the next set and detect equal one made without it
    from ai_camera_b200 import synth
    from ai_camera_b200.pipeline import BatchDetector
    det = BatchDetector(blobs[0], 2)
    synth.apply_class_bias(det.engine, bias)
    frames = [_video(540, 960, 3)[0], _video(720, 1280, 4)[0]]
    t = Table(frames, [_filter(0.45, 0.3), _filter(0.2, 0.6)])
    ref = Table(frames, [_filter(0.45, 0.3), _filter(0.2, 0.6)])
    try:
        torch.cuda.synchronize()
        before = lib.aicam_launch_count()
        for f, code in ((_filter(float("nan")), -1), (_filter(1.5), -1), (_filter(0.3, -0.5), -1),
                        (_filter(0.3, 0.5, float("inf")), -1)):
            assert lib.aicam_frame_table_set_filters(t.handle, (L.StreamFilter * 2)(_filter(0.1, 0.1), f), 2) == code
        assert lib.aicam_frame_table_set_filters(t.handle, (L.StreamFilter * 3)(*[_filter()] * 3), 3) == -4
        assert lib.aicam_frame_table_set_filters(t.handle, None, -1) == -1
        assert lib.aicam_launch_count() == before
        descs = (L.FrameDesc * 2)(*[L.FrameDesc(f.data_ptr(), None, f.shape[0], f.shape[1], f.stride(0), 0) for f in frames])
        _check(lib.aicam_frame_table_set(t.handle, descs, 2, None))
        got, want = det.detect_table(t), None
        got = [g.cpu().clone() for g in got]
        want = [w.cpu().clone() for w in det.detect_table(ref)]
        assert all(torch.equal(g, w) for g, w in zip(got, want))
    finally:
        t.close()
        ref.close()


# ---- pipeline -------------------------------------------------------------------------------------------------------

def _rows(ot, oc, on, s):
    from ai_camera_b200 import config
    return [tuple(int(v) for v in ot[s, k, :5]) + (config.CLASSES[ot[s, k, 5]], float(oc[s, k])) for k in range(on[s])]


def _pipeline(blobs, bias, n, settings=None, **kw):
    from ai_camera_b200 import synth
    from ai_camera_b200.pipeline import TrackingPipeline
    p = TrackingPipeline(blobs[0], blobs[1], n, max_tracks=128, stream_settings=settings, **kw)
    synth.apply_class_bias(p.detector.engine, bias)
    return p


def _ctor(st):
    """A StreamSettings as TrackingPipeline constructor arguments."""
    return dict(conf_threshold=st.conf_threshold, nms_threshold=st.nms_threshold, classes_to_track=st.classes_to_track,
                min_detection_confidence=st.min_detection_confidence, max_cosine_distance=st.max_cosine_distance,
                max_iou_distance=st.max_iou_distance, max_age=st.max_age, n_init=st.n_init)


def _mixed_settings():
    from ai_camera_b200.pipeline import StreamSettings
    # (the synthetic detector's tracked-class detections are people; it also finds wine glasses, which the default set
    # does not track)
    return [StreamSettings(classes_to_track={"person", "wine glass"}, n_init=2),
            StreamSettings(classes_to_track={"wine glass"}, conf_threshold=0.35, n_init=1),
            StreamSettings(nms_threshold=0.4, n_init=2),
            StreamSettings(max_age=10, n_init=1),
            StreamSettings(n_init=2),
            StreamSettings(conf_threshold=0.2, max_cosine_distance=0.3, max_iou_distance=0.6, n_init=2)]


def _to_bgr(frame):
    if frame.dim() == 3:
        return frame.contiguous()
    h, w = frame.shape[0] * 2 // 3, frame.shape[1]
    out = torch.empty((1, h, w, 3), dtype=torch.uint8, device=DEV)
    _check(_lib().aicam_nv12_to_bgr(frame.contiguous().data_ptr(), 1, h, w, out.data_ptr(), None))
    return out[0]


@gpu
def test_pipeline_streams_equal_their_reference_runs(blobs, bias):
    """Six streams of mixed sizes and kinds, one absent at some steps, each with its own settings: every stream equals a
    one-stream pipeline built with its settings as constructor arguments, and, where the settings are facade arguments,
    the YOLODetector + DeepSORT pair."""
    from ai_camera_b200 import synth
    from ai_camera_b200.deepsort_tracker import DeepSORT
    from ai_camera_b200.yolo_detector import YOLODetector
    sizes = [(540, 960), (720, 1280), (1080, 1920), (480, 640), (600, 800), (540, 960)]
    T = 8
    settings = _mixed_settings()
    videos = [_video(h, w, 110 + i, n_frames=T) for i, (h, w) in enumerate(sizes)]
    pipe = _pipeline(blobs, bias, len(sizes), settings)
    alone = [_pipeline(blobs, bias, 1, **_ctor(st)) for st in settings]
    facade = {}
    for s in (2, 3, 4, 5):  # the default classes: expressible as facade arguments
        st = settings[s]
        det = YOLODetector(blobs[0], conf_threshold=st.conf_threshold, nms_threshold=st.nms_threshold)
        synth.apply_class_bias(det.trt_engine, bias)
        facade[s] = (det, DeepSORT(blobs[1], max_cosine_distance=st.max_cosine_distance, max_iou_distance=st.max_iou_distance,
                                   max_age=st.max_age, n_init=st.n_init, max_dets=100, max_tracks=128))
    used = [0] * len(sizes)
    reported = [0] * len(sizes)
    classes = [set() for _ in sizes]
    for t in range(T):
        frames = []
        for s in range(len(sizes)):
            if s == 5 and t in (2, 5):
                frames.append(None)
                continue
            f = videos[s][used[s]]
            used[s] += 1
            frames.append(_nv12(f) if s == 4 else f)
        ot, oc, on = [x.cpu().numpy() for x in pipe.step(frames)]
        for s, f in enumerate(frames):
            if f is None:
                assert on[s] == 0
                continue
            want = _rows(*[x.cpu().numpy() for x in alone[s].step([f])], 0)
            assert _rows(ot, oc, on, s) == want, (t, s)
            reported[s] += len(want)
            classes[s] |= {r[5] for r in want}
            if s in facade:
                det, trk = facade[s]
                fb = _to_bgr(f).cpu().numpy()
                b, sc, c, _ = det.detect(fb)
                assert trk.update(b, sc, c, fb) == want, ("facade", t, s)
    assert all(r > 0 for r in reported), reported
    for s, st in enumerate(settings):  # each stream reports its own classes only
        assert classes[s] <= st.classes_to_track, (s, classes[s])
    assert not pipe.tracker.overflow().any()


@gpu
def test_neutral_settings_change_nothing(blobs, bias):
    from ai_camera_b200 import synth
    from ai_camera_b200.pipeline import StreamSettings
    S = 4
    video = synth.SynthVideo(S, (540, 960), n_frames=5, seed=17)
    plain = _pipeline(blobs, bias, S, n_init=2)
    neutral = _pipeline(blobs, bias, S, [StreamSettings(n_init=2)] * S, n_init=2)
    lib = _lib()
    for as_list in (True, False):
        for p in (plain, neutral):  # (warm: first sights of sizes and paths)
            p.step(list(video.frames(0)) if as_list else video.frames(0))
            p.tracker.reset()
        torch.cuda.synchronize()
        counts = []
        for t in range(5):
            frames = list(video.frames(t)) if as_list else video.frames(t)
            outs = []
            for p in (plain, neutral):
                before = lib.aicam_launch_count()
                outs.append([x.cpu().clone() for x in p.step(frames)])
                counts.append(lib.aicam_launch_count() - before)
            for a, b in zip(*outs):
                assert torch.equal(a, b), (as_list, t)
        assert len(set(counts)) == 1, counts
    assert neutral.launches_per_step() == plain.launches_per_step()


@gpu
def test_stacked_step_with_mixed_settings_runs_the_table(blobs, bias):
    from ai_camera_b200 import synth
    S = 6
    video = synth.SynthVideo(S, (540, 960), n_frames=5, seed=23)
    settings = _mixed_settings()
    stacked, listed = _pipeline(blobs, bias, S, settings), _pipeline(blobs, bias, S, settings)
    plain = _pipeline(blobs, bias, S, n_init=2)
    lib = _lib()
    total = 0
    for t in range(5):
        a = [x.cpu().numpy() for x in stacked.step(video.frames(t))]
        b = [x.cpu().numpy() for x in listed.step(list(video.frames(t)))]
        assert np.array_equal(a[2], b[2]), t
        for s in range(S):
            assert _rows(*a, s) == _rows(*b, s), (t, s)
        total += int(a[2].sum())
    assert total > 0
    plain.step(video.frames(0))
    torch.cuda.synchronize()
    counts = []
    for p, frames in ((stacked, video.frames(0)), (listed, list(video.frames(0))), (plain, video.frames(0))):
        before = lib.aicam_launch_count()
        p.step(frames)
        torch.cuda.synchronize()
        counts.append(lib.aicam_launch_count() - before)
    assert counts[0] == counts[1]
    assert stacked.launches_per_step() == stacked.launches_per_step(True) == plain.launches_per_step(True)
    assert counts[0] - counts[2] == stacked.launches_per_step() - plain.launches_per_step()


@gpu
def test_captured_step_follows_settings_and_presence(blobs, bias):
    from ai_camera_b200.pipeline import StreamSettings
    sizes = [(540, 960), (1080, 1920), (480, 640)]
    videos = [_video(h, w, 130 + i, n_frames=6) for i, (h, w) in enumerate(sizes)]
    masks = [[1, 1, 1], [1, 0, 1], [1, 1, 1], [0, 1, 1], [1, 1, 0], [1, 1, 1]]
    changes = {1: ([0], [StreamSettings(classes_to_track={"person"}, conf_threshold=0.45, n_init=1)]),
               3: ([1, 2], [StreamSettings(nms_threshold=0.3, max_age=2, n_init=1), StreamSettings(max_cosine_distance=0.35)]),
               4: ([0], [StreamSettings(n_init=1)])}
    g_pipe, e_pipe = (_pipeline(blobs, bias, 3, n_init=1, max_frame_hw=(1080, 1920)) for _ in range(2))
    g_pipe.step([v[0] for v in videos])
    torch.cuda.synchronize()
    g_pipe.tracker.reset()
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=stream):
        out = g_pipe.step_table()
    reported = 0
    for t in range(6):
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


@gpu
def test_resets_keep_or_take_settings(blobs, bias):
    from ai_camera_b200.aicamera_tracker import run_batched, tracks_to_rows
    from ai_camera_b200.pipeline import StreamSettings
    person = StreamSettings(classes_to_track={"person"}, conf_threshold=0.4, n_init=1, max_age=5)
    cars = StreamSettings(classes_to_track={"car", "truck", "bus", "wine glass"}, nms_threshold=0.4, n_init=2)
    sizes = [(540, 960), (720, 1280)]
    T, R = 8, 4
    videos = [_video(h, w, 150 + i, n_frames=T) for i, (h, w) in enumerate(sizes)]
    new_src = [_video(600, 800, 160 + i, n_frames=T - R) for i in range(2)]
    pipe = _pipeline(blobs, bias, 2, [person, cars])
    fresh = [_pipeline(blobs, bias, 1, **_ctor(st)) for st in (person, cars, person, person)]
    for t in range(T):
        if t == R:
            pipe.reset_streams([0])                   # keeps `person`
            pipe.reset_streams([1], settings=person)  # takes `person`
        frames = [v[t] for v in videos] if t < R else [new_src[0][t - R], new_src[1][t - R]]
        got = [x.cpu().numpy() for x in pipe.step(frames)]
        for s in range(2):
            ref = fresh[s] if t < R else fresh[2 + s]
            assert _rows(*got, s) == _rows(*[x.cpu().numpy() for x in ref.step([frames[s]])], 0), (t, s)
    assert pipe.settings == [person, person]
    # the frame loop: a refilled slot takes its source's settings in on_refill
    import cv2
    from ai_camera_b200.aicamera_tracker import video_frames
    clip = list(video_frames(CLIP, 12))
    inputs = [clip, [cv2.resize(f, (1280, 720)) for f in clip[:6]], [cv2.resize(f, (640, 480)) for f in clip[2:9]]]
    per_input = [person, cars, StreamSettings(max_age=3, n_init=1, conf_threshold=0.25)]
    from ai_camera_b200 import synth
    clip_bias = synth.shifted_class_bias(blobs[0], synth.CLIP_LOGIT_SHIFT)
    pipe = _pipeline(blobs, clip_bias, 2, per_input[:2])
    slot_input = [0, 1]
    got = [[] for _ in inputs]

    def on_refill(slot, k):
        slot_input[slot] = 2 + k
        pipe.configure_streams([slot], per_input[2 + k])

    def on_step(step, batch, table):
        tabs = [x.numpy() for x in table]
        for s, f in enumerate(batch):
            if f is not None:
                got[slot_input[s]].append(tracks_to_rows(tabs, s))
    run_batched(inputs[:2], pipe, on_step, until="all", refill=iter(inputs[2:]), on_refill=on_refill)
    total = 0
    for i, frames in enumerate(inputs):
        one = _pipeline(blobs, clip_bias, 1, **_ctor(per_input[i]))
        want = []
        run_batched([frames], one, lambda step, batch, table: want.append(tracks_to_rows([x.numpy() for x in table], 0)))
        assert got[i] == want, i
        total += sum(len(r) for r in want)
    assert total > 0


def _write_clip(path, frames):
    import cv2
    w = cv2.VideoWriter(str(path), cv2.VideoWriter_fourcc(*"mp4v"), 10, (frames[0].shape[1], frames[0].shape[0]))
    for f in frames:
        w.write(f)
    w.release()
    return str(path)


@gpu
def test_cli_runs_each_input_with_its_settings(blobs, tmp_path):
    import cv2
    from ai_camera_b200 import synth, weights
    from ai_camera_b200.aicamera_tracker import main, run_batched, tracks_to_rows, video_frames
    from ai_camera_b200.pipeline import StreamSettings, TrackingPipeline
    # a detector blob with the clip's class bias baked in (the command line takes blob paths only)
    kind, params, tensors = weights.read_blob(blobs[0])
    tensors = dict(tensors)
    for n, b in synth.shifted_class_bias(blobs[0], synth.CLIP_LOGIT_SHIFT).items():
        tensors[n + ".bias"] = b
    yolo = weights.write_blob(str(tmp_path / "yolo_clip.aicw"), kind, params, tensors)
    clip = list(video_frames(CLIP, 10))
    paths = [_write_clip(tmp_path / "a.mp4", clip), _write_clip(tmp_path / "b.mp4", [cv2.resize(f, (1280, 720)) for f in clip])]
    spec = {"default": {"n_init": 2}, "a.mp4": {"classes_to_track": ["person"], "conf_threshold": 0.4},
            "b.mp4": {"classes_to_track": ["car", "truck", "bus"], "max_age": 4, "nms_threshold": 0.4}}
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
        one = TrackingPipeline(yolo, blobs[1], 1, **_ctor(st))
        want = []
        run_batched([video_frames(p)], one, lambda step, batch, table: want.append(tracks_to_rows([x.numpy() for x in table], 0)))
        got = [[tuple(r) for r in l["tracks"]] for l in sorted((l for l in lines if l["stream"] == s), key=lambda l: l["frame"])]
        assert got == want, p
        total += sum(len(r) for r in want)
    assert total > 0
