"""Region oracle: which detections a stream with include and exclude polygons tracks, restated in numpy float32 and
plain Python integers.

The rule is that of include/aicam.h (aicam_frame_table_set_regions), which csrc/reid_crops.cu (region_kernel)
implements on the device.  A region is ``(includes, excludes)``: two lists of polygons, each a list of integer
frame-pixel ``(x, y)`` vertices.
"""
import numpy as np

from .counting import ANCHOR_LIMIT, inside


def _clamp(v):
    return max(-ANCHOR_LIMIT, min(ANCHOR_LIMIT, v))


def anchor(x1, y1, x2, y2):
    """Bottom centre of a detection box, doubled, on the integer grid: (floor(x1 + x2), floor(2 * y2)) with the sum
    rounded to float32, each clamped to [-2^24, 2^24]."""
    sx = np.float32(x1) + np.float32(x2)
    sy = np.float32(2.0) * np.float32(y2)
    return _clamp(int(np.floor(sx))), _clamp(int(np.floor(sy)))


def _doubled(points):
    return [(2 * x, 2 * y) for x, y in points]


def keep(region, box):
    """Whether a detection with ``box`` (x1, y1, x2, y2) passes ``region``: its anchor is inside some include polygon
    (or there is none) and inside no exclude polygon."""
    includes, excludes = region
    p = anchor(*box)
    if includes and not any(inside(_doubled(poly), p) for poly in includes):
        return False
    return not any(inside(_doubled(poly), p) for poly in excludes)


def keep_mask(region, boxes):
    """keep() of every row of ``boxes`` [n, 4]; all True when the region has no polygons."""
    includes, excludes = region
    if not includes and not excludes:
        return np.ones(len(boxes), bool)
    return np.array([keep(region, b) for b in boxes], bool)


def compact(region, num_dets, boxes, scores, labels):
    """One frame's detections (as detect() returns them: num_dets, boxes [K, 4], scores [K], labels [K]) without those
    the region drops, in their order and zero-padded to K: what the stream's tracker sees."""
    n = int(num_dets)
    m = np.nonzero(keep_mask(region, np.asarray(boxes[:n])))[0]
    ob, os_, ol = np.zeros_like(boxes), np.zeros_like(scores), np.zeros_like(labels)
    ob[:len(m)], os_[:len(m)], ol[:len(m)] = boxes[m], scores[m], labels[m]
    return len(m), ob, os_, ol
