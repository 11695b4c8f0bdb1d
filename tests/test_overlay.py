"""Overlay (N3), CPU side: the oracle compositor is pinned to OpenCV and to the reference's own drawing functions
(src/utils/visualization.py), and the decal builder of ai-camera_b200/visualization.py is checked through it."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
cv2 = pytest.importorskip("cv2")
from ai_camera_b200 import config, visualization as V  # noqa: E402
from oracle import overlay as O  # noqa: E402
from oracle import ref_bridge  # noqa: E402


def reference_visualization():
    if not ref_bridge.available():
        pytest.skip("needs oracle/_ref, a snapshot of the original AI-Camera sources (python oracle/build_ref.py "
                    "<checkout of the original project>); no recorded output of its drawing functions replaces it")
    ref_bridge.import_reference()
    import src.utils.visualization as rv
    rv.config.CLASS_COLORS = dict(config.CLASS_COLORS)  # (the reference draws its colours at random at import)
    return rv


def random_rects(rng, n, H, W):
    out = [(4, 3, 12, 9), (4, 3, 6, 5), (4, 3, 5, 4), (4, 3, 4, 3), (-1, -1, 5, 5), (4, 3, W + 12, 9), (12, 9, 4, 3),
           (0, 0, W - 1, H - 1), (-20, -20, -5, -5), (W - 2, H - 2, W + 5, H + 5), (3, 5, 3, 20), (3, 5, 30, 5)]
    for _ in range(n):
        x1, x2 = rng.integers(-10, W + 10, 2)
        y1, y2 = rng.integers(-10, H + 10, 2)
        out.append((int(x1), int(y1), int(x2), int(y2)))
    return out


@pytest.mark.parametrize("thickness,typ", [(2, 0), (-1, 1)])
def test_rectangles_match_cv2(thickness, typ):
    rng = np.random.default_rng(3)
    H, W = 48, 64
    for (x1, y1, x2, y2) in random_rects(rng, 300, H, W):
        ref = np.zeros((H, W, 3), np.uint8)
        cv2.rectangle(ref, (x1, y1), (x2, y2), (10, 200, 77), thickness)
        got = O.draw_items(np.zeros((H, W, 3), np.uint8), [(typ, x1, y1, x2, y2, 10 | 200 << 8 | 77 << 16, 0)], None)
        assert np.array_equal(ref, got), (x1, y1, x2, y2)


def tracks_case(rng, H, W, n):
    objs = []
    for i in range(n):
        x1 = int(rng.integers(-20, W - 40)); y1 = int(rng.integers(-10, H - 40))
        x2 = x1 + int(rng.integers(20, 300)); y2 = y1 + int(rng.integers(30, 400))
        name = ["person", "car", "bus", "truck", "motorcycle"][int(rng.integers(0, 5))]
        objs.append((x1, y1, x2, y2, int(rng.integers(1, 5000)), name) + ((float(rng.random()),) if i % 3 == 0 else ()))
    return objs


def check_close(got, ref, max_diff=2, max_frac=2e-3):
    d = np.abs(got.astype(np.int16) - ref.astype(np.int16))
    assert d.max() <= max_diff, "max difference %d" % d.max()
    assert (d != 0).any(-1).mean() <= max_frac, "differing pixels %.5f" % (d != 0).any(-1).mean()
    return int(d.max()), 100 * float((d != 0).any(-1).mean())


def test_track_overlay_matches_reference_drawing():
    rv = reference_visualization()
    rng = np.random.default_rng(11)
    H, W = 540, 960
    ov = V.Overlay(device="cpu", slots=64)
    worst = (0, 0.0)
    for trial in range(4):
        frame = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
        objs = tracks_case(rng, H, W, 12)
        ref = rv.draw_tracks(frame.copy(), objs)
        got = O.draw_items(frame.copy(), ov.track_items(objs, (H, W)), ov.atlas.numpy())
        worst = max(worst, check_close(got, ref))
    print("track overlay vs reference: max difference %d grey levels, %.4f %% of the pixels differ" % worst)


def test_detection_overlay_matches_reference_drawing():
    rv = reference_visualization()
    rng = np.random.default_rng(12)
    H, W = 360, 640
    ov = V.Overlay(device="cpu", slots=64)
    frame = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    boxes = np.array([[30.7, 40.2, 200.9, 300.1], [300, 20, 420, 200], [500, 100, 630, 350]], np.float32)
    scores = np.array([0.91, 0.456, 0.3], np.float32)
    cls = np.array([0, 2, 99])
    ref = rv.draw_detections(frame.copy(), boxes, scores, cls, config.CLASSES)
    got = O.draw_items(frame.copy(), ov.detection_items(boxes, scores, cls, config.CLASSES, (H, W)), ov.atlas.numpy())
    check_close(got, ref)


def test_panels_match_reference_drawing():
    rv = reference_visualization()
    rng = np.random.default_rng(13)
    H, W = 360, 960
    frame = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    lines = ["AICamera: YOLOv8 + DeepSORT", "Input: aicamera_test_clip.mp4", "FPS: 29.97"]
    ref = rv.draw_info_panel(frame.copy(), lines)
    decal, (w, h) = V._affine_decal(lambda img: V.Overlay._draw_info_panel(img, lines), 192, 1024)
    got = O.draw_items(frame.copy(), [(2, 0, 0, w, h, 0, 0)], decal[None])
    # the panel's text is wider than its grey background in places: strokes that overlap OUTSIDE a filled background
    # are blended twice by cv2's integer arithmetic, which one affine map per pixel only follows to a few grey levels
    print("info panel vs reference: max difference %d, %.4f %% of the pixels differ" % check_close(got, ref, max_diff=6))
    ref = rv.draw_fps(frame.copy(), 123.456)
    decal, (w, h) = V._affine_decal(lambda img: V.Overlay._draw_fps(img, 123.456), 192, 1024)
    got = O.draw_items(frame.copy(), [(2, 0, 0, w, h, 0, 0)], decal[None])
    print("fps box vs reference: max difference %d, %.4f %% of the pixels differ" % check_close(got, ref, max_diff=6))


def test_label_cache_reuses_and_evicts_slots():
    ov = V.Overlay(device="cpu", slots=3)
    a = ov.track_items([(10, 50, 60, 90, 1, "person")], (540, 960))
    b = ov.track_items([(30, 70, 80, 120, 1, "person")], (540, 960))
    assert a[1][6] == b[1][6] and len(ov._cache) == 1  # same label text: same slot
    for i in range(2, 6):
        ov.track_items([(10, 50, 60, 90, i, "car")], (540, 960))
    assert len(ov._cache) == 3 and len({v[0] for v in ov._cache.values()}) == 3
